// ffi.cpp -- the C ABI: every symbol of include/sourmash.h (the reference's src/ffi.rs,
// src/utils.rs, src/errors.rs surface) plus the batch extension of include/sourmash_b200.h.
//
// Error convention of the reference's `ffi_fn!` / `landingpad` (src/utils.rs:18-45,154-166):
// the body runs inside a catch-all; an error is stored in a thread-local slot and the call
// returns an all-zero value.  Here the catch-all is try/catch and the slot holds (code, message).
// The reference leaves some entry points unwrapped (they assert on NULL and abort); this build
// wraps all of them, which only adds recorded errors where the reference would have aborted.
#include <algorithm>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <new>
#include <string>
#include <vector>

#include "../../include/sourmash_b200.h"
#include "collection.hpp"
#include "comm.hpp"
#include "kernels.cuh"
#include "minhash.hpp"
#include "nodegraph.hpp"
#include "signature.hpp"

using smb200::SourmashError;
typedef smb200::KmerMinHash MH;
typedef smb200::Signature SIG;
typedef smb200::SketchCollection COLL;
typedef smb200::Nodegraph NG;

namespace {

struct LastError {
    uint32_t code = 0;
    std::string message;
};
thread_local LastError g_last_error;

// Locking (SURVEY 8(b) Threading; utils.rs:14-16): there is no library-wide lock.  Every host thread has its own
// stream and scratch (device.cu), the error slot is thread-local, and a call holds only the locks of the objects
// it is handed -- so distinct handles are independent, as in the reference, and host-only calls (hash_murmur,
// the scalar getters, string helpers) take no lock at all.  The per-object lock makes concurrent calls on ONE
// handle safe as well (the reference's &self methods may be shared between threads; here even a read can
// flush deferred work, i.e. mutate).
typedef std::mutex Mu;
struct Guard {  // locks up to two objects (the same object twice: once), in address order
    Mu *a = nullptr, *b = nullptr;
    explicit Guard(Mu &x) : a(&x) { a->lock(); }
    Guard(Mu &x, Mu &y) : a(&x), b(&y) {
        if (a == b) b = nullptr;
        else if (b < a) std::swap(a, b);
        a->lock();
        if (b) b->lock();
    }
    ~Guard() {
        if (b) b->unlock();
        a->unlock();
    }
    Guard(const Guard &) = delete;
    Guard &operator=(const Guard &) = delete;
};
struct GuardN {  // any number of objects
    std::vector<Mu *> ms;
    void add(Mu &m) { ms.push_back(&m); }
    void lock() {
        std::sort(ms.begin(), ms.end());
        ms.erase(std::unique(ms.begin(), ms.end()), ms.end());
        for (Mu *m : ms) m->lock();
        locked = true;
    }
    ~GuardN() {
        if (locked) for (size_t i = ms.size(); i-- > 0;) ms[i]->unlock();
    }
    bool locked = false;
};

void set_error(uint32_t code, const std::string &msg) {
    g_last_error.code = code;
    g_last_error.message = msg;
}

template <class T, class F>
T landingpad(F &&body) {
    try {
        return body();
    } catch (const SourmashError &e) {
        set_error(e.code, e.what());
    } catch (const std::bad_alloc &) {
        set_error(smb200::ERR_PANIC, "sourmash panicked: out of memory");
    } catch (const std::exception &e) {
        set_error(smb200::ERR_PANIC, std::string("sourmash panicked: ") + e.what());
    } catch (...) {
        set_error(smb200::ERR_PANIC, "sourmash panicked: unknown exception");
    }
    return T();
}
template <class F>
void landingpad_void(F &&body) {
    landingpad<int>([&]() { body(); return 0; });
}

[[noreturn]] void panic(const std::string &what) { throw SourmashError(smb200::ERR_PANIC, "sourmash panicked: " + what); }

template <class T>
T *nonnull(T *p, const char *what) {
    if (!p) panic(std::string("assertion failed: !") + what + ".is_null()");
    return p;
}
MH *mh(KmerMinHash *p) { return reinterpret_cast<MH *>(nonnull(p, "ptr")); }
MH *mh(const KmerMinHash *p) { return reinterpret_cast<MH *>(const_cast<KmerMinHash *>(nonnull(p, "other"))); }
SIG *sig(Signature *p) { return reinterpret_cast<SIG *>(nonnull(p, "ptr")); }
COLL *coll(SketchCollection *p) { return reinterpret_cast<COLL *>(nonnull(p, "collection")); }
NG *ngp(Nodegraph *p) { return reinterpret_cast<NG *>(nonnull(p, "nodegraph")); }

SourmashStr str_from(const std::string &s) {  // SourmashStr::from_string, utils.rs:194-204
    SourmashStr r;
    r.len = s.size();
    r.data = static_cast<char *>(malloc(s.size() ? s.size() : 1));
    if (!r.data) throw std::bad_alloc();
    memcpy(r.data, s.data(), s.size());
    r.owned = true;
    return r;
}
SourmashStr str_empty() {
    SourmashStr r;
    r.data = nullptr; r.len = 0; r.owned = false;
    return r;
}
bool valid_utf8(const char *s) {
    const unsigned char *p = reinterpret_cast<const unsigned char *>(s);
    while (*p) {
        int n = (*p < 0x80) ? 0 : ((*p >> 5) == 6 ? 1 : ((*p >> 4) == 14 ? 2 : ((*p >> 3) == 30 ? 3 : -1)));
        if (n < 0) return false;
        p++;
        for (; n > 0; n--, p++) if ((*p >> 6) != 2) return false;
    }
    return true;
}
uint64_t *copy_out(const std::vector<uint64_t> &v) {  // Box<[u64]> handed to the caller
    uint64_t *out = static_cast<uint64_t *>(malloc(v.size() ? v.size() * 8 : 8));
    if (!out) throw std::bad_alloc();
    if (!v.empty()) memcpy(out, v.data(), v.size() * 8);
    return out;
}

}  // namespace

extern "C" {

// ---------------------------------------------------------------------------------------------
// hashing, lifecycle
// ---------------------------------------------------------------------------------------------
uint64_t hash_murmur(const char *kmer, uint64_t seed) {
    return landingpad<uint64_t>([&]() {
        nonnull(kmer, "kmer");
        return smb200::hash_murmur_host(reinterpret_cast<const uint8_t *>(kmer), strlen(kmer), seed);
    });
}

KmerMinHash *kmerminhash_new(uint32_t n, uint32_t k, bool prot, uint64_t seed, uint64_t mx, bool track_abundance) {
    return landingpad<KmerMinHash *>([&]() { return reinterpret_cast<KmerMinHash *>(new MH(n, k, prot, seed, mx, track_abundance)); });
}
void kmerminhash_free(KmerMinHash *ptr) {
    if (!ptr) return;
    landingpad_void([&]() { delete reinterpret_cast<MH *>(ptr); });
}

// ---------------------------------------------------------------------------------------------
// ingest
// ---------------------------------------------------------------------------------------------
void kmerminhash_add_sequence(KmerMinHash *ptr, const char *sequence, bool force) {
    landingpad_void([&]() {
        MH *m = mh(ptr);
        nonnull(sequence, "sequence");
        Guard lk(m->mu);
        m->add_sequence(reinterpret_cast<const uint8_t *>(sequence), strlen(sequence), force);
    });
}
void kmerminhash_add_hash(KmerMinHash *ptr, uint64_t h) {
    landingpad_void([&]() { MH *m = mh(ptr); Guard lk(m->mu); m->add_hash(h); });
}
void kmerminhash_add_word(KmerMinHash *ptr, const char *word) {
    landingpad_void([&]() {
        MH *m = mh(ptr);
        nonnull(word, "word");
        Guard lk(m->mu);
        m->add_word(reinterpret_cast<const uint8_t *>(word), strlen(word));
    });
}
void kmerminhash_add_from(KmerMinHash *ptr, const KmerMinHash *other) {
    landingpad_void([&]() { MH *a = mh(ptr), *b = mh(other); Guard lk(a->mu, b->mu); a->add_from(*b); });
}
void kmerminhash_mins_push(KmerMinHash *ptr, uint64_t val) {
    landingpad_void([&]() { MH *m = mh(ptr); Guard lk(m->mu); m->mins_push(val); });
}
void kmerminhash_abunds_push(KmerMinHash *ptr, uint64_t val) {
    landingpad_void([&]() { MH *m = mh(ptr); Guard lk(m->mu); m->abunds_push(val); });
}

// ---------------------------------------------------------------------------------------------
// combine / compare
// ---------------------------------------------------------------------------------------------
void kmerminhash_merge(KmerMinHash *ptr, const KmerMinHash *other) {
    landingpad_void([&]() { MH *a = mh(ptr), *b = mh(other); Guard lk(a->mu, b->mu); a->merge(*b); });
}
double kmerminhash_compare(KmerMinHash *ptr, const KmerMinHash *other) {
    return landingpad<double>([&]() { MH *a = mh(ptr), *b = mh(other); Guard lk(a->mu, b->mu); return a->compare(*b); });
}
uint64_t kmerminhash_count_common(KmerMinHash *ptr, const KmerMinHash *other) {
    return landingpad<uint64_t>([&]() { MH *a = mh(ptr), *b = mh(other); Guard lk(a->mu, b->mu); return a->count_common(*b); });
}
uint64_t kmerminhash_intersection(KmerMinHash *ptr, const KmerMinHash *other) {
    return landingpad<uint64_t>([&]() -> uint64_t {
        MH *a = mh(ptr), *b = mh(other);
        Guard lk(a->mu, b->mu);
        try {
            return a->intersection_size(*b).second;
        } catch (const SourmashError &e) {
            // ffi.rs:304-307: `if let Ok(..)` swallows the compatibility error and yields 0
            if (e.code >= smb200::ERR_MISMATCH_KSIZES && e.code <= smb200::ERR_MISMATCH_SEED) return 0;
            throw;
        }
    });
}

// ---------------------------------------------------------------------------------------------
// read-out
// ---------------------------------------------------------------------------------------------
const uint64_t *kmerminhash_get_mins(KmerMinHash *ptr) {
    return landingpad<const uint64_t *>([&]() { MH *m = mh(ptr); Guard lk(m->mu); return (const uint64_t *)copy_out(m->mins()); });
}
const uint64_t *kmerminhash_get_abunds(KmerMinHash *ptr) {
    return landingpad<const uint64_t *>([&]() -> const uint64_t * {
        MH *m = mh(ptr);
        Guard lk(m->mu);
        if (!m->track_abundance()) return nullptr;
        return copy_out(m->abunds());
    });
}
uintptr_t kmerminhash_get_mins_size(KmerMinHash *ptr) {
    return landingpad<uintptr_t>([&]() { MH *m = mh(ptr); Guard lk(m->mu); return (uintptr_t)m->size(); });
}
uintptr_t kmerminhash_get_abunds_size(KmerMinHash *ptr) {
    return landingpad<uintptr_t>([&]() -> uintptr_t {
        MH *m = mh(ptr);
        Guard lk(m->mu);
        return m->track_abundance() ? m->abunds().size() : 0;
    });
}
uint64_t kmerminhash_get_min_idx(KmerMinHash *ptr, uint64_t idx) {
    return landingpad<uint64_t>([&]() {
        MH *m = mh(ptr);
        Guard lk(m->mu);
        const std::vector<uint64_t> &v = m->mins();
        if (idx >= v.size()) panic("index out of bounds: the len is " + std::to_string(v.size()) + " but the index is " + std::to_string(idx));
        return v[idx];
    });
}
uint64_t kmerminhash_get_abund_idx(KmerMinHash *ptr, uint64_t idx) {
    return landingpad<uint64_t>([&]() -> uint64_t {
        MH *m = mh(ptr);
        Guard lk(m->mu);
        if (!m->track_abundance()) return 0;  // ffi.rs:161-163
        const std::vector<uint64_t> &v = m->abunds();
        if (idx >= v.size()) panic("index out of bounds: the len is " + std::to_string(v.size()) + " but the index is " + std::to_string(idx));
        return v[idx];
    });
}
bool kmerminhash_is_protein(KmerMinHash *ptr) { return landingpad<bool>([&]() { return mh(ptr)->is_protein; }); }
uint64_t kmerminhash_seed(KmerMinHash *ptr) { return landingpad<uint64_t>([&]() { return mh(ptr)->seed; }); }
bool kmerminhash_track_abundance(KmerMinHash *ptr) { return landingpad<bool>([&]() { MH *m = mh(ptr); Guard lk(m->mu); return m->track_abundance(); }); }
uint32_t kmerminhash_num(KmerMinHash *ptr) { return landingpad<uint32_t>([&]() { return mh(ptr)->num; }); }
uint32_t kmerminhash_ksize(KmerMinHash *ptr) { return landingpad<uint32_t>([&]() { return mh(ptr)->ksize; }); }
uint64_t kmerminhash_max_hash(KmerMinHash *ptr) { return landingpad<uint64_t>([&]() { return mh(ptr)->max_hash; }); }

// ---------------------------------------------------------------------------------------------
// Signature
// ---------------------------------------------------------------------------------------------
Signature *signature_new(void) {
    return landingpad<Signature *>([&]() { return reinterpret_cast<Signature *>(new SIG()); });
}
void signature_free(Signature *ptr) {
    if (!ptr) return;
    landingpad_void([&]() { delete reinterpret_cast<SIG *>(ptr); });
}
void signature_set_name(Signature *ptr, const char *name) {
    landingpad_void([&]() {
        SIG *s = sig(ptr);
        nonnull(name, "name");
        Guard lk(s->mu);
        if (valid_utf8(name)) { s->has_name = true; s->name = name; }  // ffi.rs:356-359: ignored when not UTF-8
    });
}
void signature_set_filename(Signature *ptr, const char *name) {
    landingpad_void([&]() {
        SIG *s = sig(ptr);
        nonnull(name, "name");
        Guard lk(s->mu);
        if (valid_utf8(name)) { s->has_filename = true; s->filename = name; }
    });
}
void signature_push_mh(Signature *ptr, const KmerMinHash *other) {
    landingpad_void([&]() { SIG *s = sig(ptr); MH *m = mh(other); Guard lk(s->mu, m->mu); s->signatures.emplace_back(m->clone()); });
}
void signature_set_mh(Signature *ptr, const KmerMinHash *other) {
    landingpad_void([&]() {
        SIG *s = sig(ptr);
        MH *m = mh(other);
        Guard lk(s->mu, m->mu);
        std::unique_ptr<MH> c(m->clone());
        s->signatures.clear();
        s->signatures.push_back(std::move(c));
    });
}
SourmashStr signature_get_name(Signature *ptr) {
    return landingpad<SourmashStr>([&]() { SIG *s = sig(ptr); Guard lk(s->mu); return str_from(s->has_name ? s->name : std::string()); });
}
SourmashStr signature_get_filename(Signature *ptr) {
    return landingpad<SourmashStr>([&]() { SIG *s = sig(ptr); Guard lk(s->mu); return str_from(s->has_filename ? s->filename : std::string()); });
}
SourmashStr signature_get_license(Signature *ptr) {
    return landingpad<SourmashStr>([&]() { SIG *s = sig(ptr); Guard lk(s->mu); return str_from(s->license); });
}
KmerMinHash *signature_first_mh(Signature *ptr) {
    return landingpad<KmerMinHash *>([&]() {
        SIG *s = sig(ptr);
        Guard lk(s->mu);
        MH *out = s->signatures.empty() ? MH::make_default() : s->signatures[0]->clone();  // ffi.rs:466-471
        return reinterpret_cast<KmerMinHash *>(out);
    });
}
KmerMinHash **signature_get_mhs(Signature *ptr, uintptr_t *size) {
    return landingpad<KmerMinHash **>([&]() {
        SIG *s = sig(ptr);
        nonnull(size, "size");
        Guard lk(s->mu);
        const size_t n = s->signatures.size();
        KmerMinHash **arr = static_cast<KmerMinHash **>(malloc((n ? n : 1) * sizeof(KmerMinHash *)));
        if (!arr) throw std::bad_alloc();
        for (size_t i = 0; i < n; i++) arr[i] = reinterpret_cast<KmerMinHash *>(s->signatures[i]->clone());
        *size = n;
        return arr;
    });
}
bool signature_eq(Signature *ptr, Signature *other) {
    return landingpad<bool>([&]() { SIG *a = sig(ptr), *b = sig(other); Guard lk(a->mu, b->mu); return a->equals(*b); });
}
SourmashStr signature_save_json(Signature *ptr) {
    return landingpad<SourmashStr>([&]() {
        std::string out;
        SIG *s = sig(ptr);
        Guard lk(s->mu);
        s->to_json(out);
        return str_from(out);
    });
}
SourmashStr signatures_save_buffer(Signature **ptr, uintptr_t size) {
    return landingpad<SourmashStr>([&]() {
        nonnull(ptr, "ptr");
        GuardN lk;
        for (uintptr_t i = 0; i < size; i++) lk.add(sig(ptr[i])->mu);
        lk.lock();
        SourmashStr r;
        size_t len = 0;
        r.data = smb200::signatures_to_json(reinterpret_cast<SIG *const *>(ptr), size, &len);
        r.len = len;
        r.owned = true;
        return r;
    });
}
static Signature **hand_over(std::vector<std::unique_ptr<SIG>> &sigs, uintptr_t *size) {
    const size_t n = sigs.size();
    Signature **arr = static_cast<Signature **>(malloc((n ? n : 1) * sizeof(Signature *)));
    if (!arr) throw std::bad_alloc();
    for (size_t i = 0; i < n; i++) arr[i] = reinterpret_cast<Signature *>(sigs[i].release());
    *size = n;
    return arr;
}
Signature **signatures_load_path(const char *ptr, bool ignore_md5sum, uintptr_t ksize, const char *select_moltype,
                                 uintptr_t *size) {
    (void)ignore_md5sum;  // ffi.rs:555 "TODO: implement ignore_md5sum"
    return landingpad<Signature **>([&]() {
        nonnull(ptr, "ptr");
        nonnull(size, "size");
        if (select_moltype && !valid_utf8(select_moltype)) throw SourmashError(smb200::ERR_UNKNOWN, "invalid utf-8 in select_moltype");
        std::vector<std::unique_ptr<SIG>> sigs = smb200::load_signatures_path(ptr, ksize, select_moltype);
        return hand_over(sigs, size);
    });
}
Signature **signatures_load_buffer(const char *ptr, uintptr_t insize, bool ignore_md5sum, uintptr_t ksize,
                                   const char *select_moltype, uintptr_t *size) {
    (void)ignore_md5sum;
    return landingpad<Signature **>([&]() {
        nonnull(ptr, "ptr");
        nonnull(size, "size");
        if (select_moltype && !valid_utf8(select_moltype)) throw SourmashError(smb200::ERR_UNKNOWN, "invalid utf-8 in select_moltype");
        std::vector<std::unique_ptr<SIG>> sigs = smb200::load_signatures(ptr, insize, ksize, select_moltype);
        return hand_over(sigs, size);
    });
}

// ---------------------------------------------------------------------------------------------
// errors and strings
// ---------------------------------------------------------------------------------------------
void sourmash_init(void) {}  // the reference installs its panic hook here; nothing to install
void sourmash_err_clear(void) { g_last_error.code = 0; g_last_error.message.clear(); }
SourmashErrorCode sourmash_err_get_last_code(void) { return g_last_error.code; }
SourmashStr sourmash_err_get_last_message(void) {
    if (g_last_error.code == 0) return str_empty();
    try { return str_from(g_last_error.message); } catch (...) { return str_empty(); }
}
SourmashStr sourmash_err_get_backtrace(void) { return str_empty(); }
void sourmash_str_free(SourmashStr *s) {
    if (!s || !s->owned) return;
    free(s->data);
    s->data = nullptr; s->len = 0; s->owned = false;
}
SourmashStr sourmash_str_from_cstr(const char *s) {
    return landingpad<SourmashStr>([&]() {
        nonnull(s, "s");
        if (!valid_utf8(s)) throw SourmashError(smb200::ERR_UNKNOWN, "invalid utf-8 sequence");
        return str_from(std::string(s));
    });
}

// ---------------------------------------------------------------------------------------------
// extension (include/sourmash_b200.h)
// ---------------------------------------------------------------------------------------------
void smgpu_set_device(int32_t device) {
    landingpad_void([&]() { smb200::set_requested_device(device); });
}
int32_t smgpu_device(int32_t *sm_count) {
    return landingpad<int32_t>([&]() {
        smb200::Context &ctx = smb200::Context::get();
        if (sm_count) *sm_count = ctx.sm_count;
        return (int32_t)ctx.device;
    });
}
uint64_t smgpu_launch_count(void) { return smb200::g_launch_count.load(); }
uint64_t smgpu_stream(void) {
    return landingpad<uint64_t>([&]() { return (uint64_t)reinterpret_cast<uintptr_t>(smb200::Context::get().stream); });
}
void smgpu_profile_enable(bool on) { smb200::prof_enable(on); }
void smgpu_profile_read(int32_t kind, double *ms, uint64_t *launches, bool reset) {
    landingpad_void([&]() { smb200::prof_read(kind, ms, launches, reset); });
}
double smgpu_int_peak(int32_t mode, int32_t iters, int32_t blocks) {
    return landingpad<double>([&]() {
        smb200::Context &ctx = smb200::Context::get();
        ctx.misc[0].reserve(4096);
        cudaEvent_t e0, e1;
        SM_CUDA(cudaEventCreate(&e0));
        SM_CUDA(cudaEventCreate(&e1));
        smb200::launch_int_peak(ctx.misc[0].as<uint32_t>(), 16, blocks, mode, ctx.stream);  // warm
        SM_CUDA(cudaEventRecord(e0, ctx.stream));
        smb200::launch_int_peak(ctx.misc[0].as<uint32_t>(), iters, blocks, mode, ctx.stream);
        SM_CUDA(cudaEventRecord(e1, ctx.stream));
        SM_CUDA(cudaEventSynchronize(e1));
        float ms = 0;
        SM_CUDA(cudaEventElapsedTime(&ms, e0, e1));
        cudaEventDestroy(e0);
        cudaEventDestroy(e1);
        // 8 chains x 8 unrolled steps per iteration, one instruction each (mode 2: 4 IMAD + 4 LOP3/SHF pairs)
        const double instr = (double)iters * 64.0 * 256.0 * (double)blocks;
        return instr / (ms * 1e-3);
    });
}
void *smgpu_alloc_pinned(uintptr_t bytes) {
    return landingpad<void *>([&]() {
        smb200::Context::get();
        void *p = nullptr;
        SM_CUDA(cudaMallocHost(&p, bytes ? bytes : 1));
        return p;
    });
}
void smgpu_free_pinned(void *ptr) {
    if (ptr) cudaFreeHost(ptr);
}
void kmerminhash_slice_free(const uint64_t *ptr) { free(const_cast<uint64_t *>(ptr)); }

// north_star's names for the two similarity measures (the crate itself calls them compare and Leaf::containment)
double kmerminhash_jaccard(KmerMinHash *ptr, const KmerMinHash *other) { return kmerminhash_compare(ptr, other); }
double kmerminhash_containment(KmerMinHash *ptr, const KmerMinHash *other) {
    return landingpad<double>([&]() { MH *a = mh(ptr), *b = mh(other); Guard lk(a->mu, b->mu); return a->containment(*b); });
}
const uint64_t *kmerminhash_intersection_hashes(KmerMinHash *ptr, const KmerMinHash *other, uintptr_t *n_common, uint64_t *size) {
    return landingpad<const uint64_t *>([&]() {
        MH *a = mh(ptr), *b = mh(other);
        nonnull(n_common, "n_common");
        Guard lk(a->mu, b->mu);
        std::pair<std::vector<uint64_t>, uint64_t> r = a->intersection(*b);
        *n_common = r.first.size();
        if (size) *size = r.second;
        return (const uint64_t *)copy_out(r.first);
    });
}

void kmerminhash_add_sequences(KmerMinHash *const *mhs, uintptr_t n_mhs, const char *buf, const uint64_t *offsets,
                               uint64_t n_seqs, bool force, bool on_device) {
    landingpad_void([&]() {
        nonnull(mhs, "mhs");
        nonnull(offsets, "offsets");
        if (n_seqs == 0) return;
        nonnull(buf, "buf");
        smb200::SeqBatch b;
        b.buf = reinterpret_cast<const uint8_t *>(buf);
        b.offsets = offsets;
        b.n_seqs = n_seqs;
        b.on_device = on_device;
        if (on_device) {
            uint64_t last = 0;
            smb200::Context &ctx = smb200::Context::get();
            SM_CUDA(cudaMemcpyAsync(&last, offsets + n_seqs, 8, cudaMemcpyDeviceToHost, ctx.stream));
            ctx.sync();
            b.n_bytes = last;
        } else {
            if (offsets[0] != 0) smb200::throw_internal("offsets[0] must be 0");
            b.n_bytes = offsets[n_seqs];
        }
        GuardN lk;
        for (uintptr_t i = 0; i < n_mhs; i++) lk.add(mh(mhs[i])->mu);
        lk.lock();
        MH::add_sequences(reinterpret_cast<MH *const *>(mhs), (int)n_mhs, b, force);
    });
}
void kmerminhash_add_reads(KmerMinHash *const *mhs, uintptr_t n_mhs, const char *buf, uint64_t n_reads, uint32_t read_len,
                           bool force, bool on_device) {
    landingpad_void([&]() {
        nonnull(mhs, "mhs");
        if (n_reads == 0 || read_len == 0) return;
        nonnull(buf, "buf");
        smb200::SeqBatch b;
        b.buf = reinterpret_cast<const uint8_t *>(buf);
        b.n_seqs = n_reads;
        b.read_len = read_len;
        b.n_bytes = n_reads * (uint64_t)read_len;
        b.on_device = on_device;
        GuardN lk;
        for (uintptr_t i = 0; i < n_mhs; i++) lk.add(mh(mhs[i])->mu);
        lk.lock();
        MH::add_sequences(reinterpret_cast<MH *const *>(mhs), (int)n_mhs, b, force);
    });
}
void kmerminhash_add_reads_2bit(KmerMinHash *const *mhs, uintptr_t n_mhs, const uint8_t *packed, uint64_t n_reads, uint32_t read_len,
                                bool on_device) {
    landingpad_void([&]() {
        nonnull(mhs, "mhs");
        if (n_reads == 0 || read_len == 0) return;
        nonnull(packed, "packed");
        smb200::SeqBatch b;
        b.packed2 = packed;
        b.n_seqs = n_reads;
        b.read_len = read_len;
        b.n_bytes = n_reads * (uint64_t)read_len;
        b.on_device = on_device;
        GuardN lk;
        for (uintptr_t i = 0; i < n_mhs; i++) lk.add(mh(mhs[i])->mu);
        lk.lock();
        MH::add_sequences(reinterpret_cast<MH *const *>(mhs), (int)n_mhs, b, true);   // every base is one of ACGT: nothing can fail
    });
}
void kmerminhash_set_mins(KmerMinHash *ptr, const uint64_t *mins, uintptr_t n, const uint64_t *abunds, uintptr_t n_abunds) {
    landingpad_void([&]() {
        MH *m = mh(ptr);
        if (n) nonnull(mins, "mins");
        Guard lk(m->mu);
        m->set_from_host(mins, n, m->track_abundance() ? abunds : nullptr, abunds ? n_abunds : 0);
    });
}
uintptr_t kmerminhash_copy_mins(KmerMinHash *ptr, uint64_t *mins, uint64_t *abunds, bool on_device) {
    return landingpad<uintptr_t>([&]() -> uintptr_t {
        MH *m = mh(ptr);
        Guard lk(m->mu);
        size_t n = 0, na = 0;
        const uint64_t *dm = m->device_mins(&n);
        const uint64_t *da = m->device_abunds(&na);
        smb200::Context &ctx = smb200::Context::get();
        const cudaMemcpyKind kind = on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost;
        if (mins && n) SM_CUDA(cudaMemcpyAsync(mins, dm, n * 8, kind, ctx.stream));
        if (abunds && da && na) SM_CUDA(cudaMemcpyAsync(abunds, da, na * 8, kind, ctx.stream));
        ctx.sync();
        return n;
    });
}
SourmashStr kmerminhash_md5sum(KmerMinHash *ptr) {
    return landingpad<SourmashStr>([&]() { MH *m = mh(ptr); Guard lk(m->mu); return str_from(m->md5sum()); });
}

SketchCollection *smgpu_collection_new(void) {
    return landingpad<SketchCollection *>([&]() { return reinterpret_cast<SketchCollection *>(new COLL()); });
}
void smgpu_collection_free(SketchCollection *c) {
    if (!c) return;
    landingpad_void([&]() { delete reinterpret_cast<COLL *>(c); });
}
void smgpu_collection_push(SketchCollection *c, KmerMinHash *m) {
    landingpad_void([&]() { COLL *cc = coll(c); MH *s = mh(m); Guard lk(cc->mu, s->mu); cc->push(*s); });
}
void smgpu_collection_push_signatures(SketchCollection *c, Signature *const *sigs, uintptr_t n) {
    landingpad_void([&]() {
        COLL *cc = coll(c);
        if (n) nonnull(sigs, "sigs");
        GuardN lk;
        lk.add(cc->mu);
        for (uintptr_t i = 0; i < n; i++) lk.add(sig(sigs[i])->mu);
        lk.lock();
        size_t extra = 0;
        for (uintptr_t i = 0; i < n; i++) {
            SIG *s = sig(sigs[i]);
            if (s->signatures.empty())
                throw SourmashError(smb200::ERR_PANIC, "sourmash panicked: index out of bounds: the len is 0 but the index is 0");
            extra += s->signatures[0]->mins().size();
        }
        cc->h_hashes.reserve(cc->h_hashes.size() + extra);
        cc->h_offsets.reserve(cc->h_offsets.size() + n);
        cc->h_nums.reserve(cc->h_nums.size() + n);
        for (uintptr_t i = 0; i < n; i++) cc->push(*sig(sigs[i])->signatures[0]);
    });
}
SketchCollection *smgpu_collection_from_csr(const uint64_t *hashes, const uint64_t *offsets, uint64_t n_rows, uint32_t num,
                                            uint32_t ksize, uint64_t seed, uint64_t max_hash, bool on_device) {
    return landingpad<SketchCollection *>([&]() {
        nonnull(offsets, "offsets");
        return reinterpret_cast<SketchCollection *>(COLL::from_csr(hashes, offsets, n_rows, num, ksize, seed, max_hash, on_device));
    });
}
SketchCollection *smgpu_sketch_collection(const char *buf, const uint64_t *offsets, uint64_t n_seqs, uint32_t num, uint32_t ksize,
                                          uint64_t seed, uint64_t max_hash, bool on_device) {
    return landingpad<SketchCollection *>([&]() {
        if (n_seqs) { nonnull(offsets, "offsets"); }
        return reinterpret_cast<SketchCollection *>(smb200::sketch_collection(reinterpret_cast<const uint8_t *>(buf), offsets, n_seqs, num,
                                                                              ksize, seed, max_hash, on_device));
    });
}
void smgpu_sketch_collections(const char *buf, const uint64_t *offsets, uint64_t n_seqs, KmerMinHash *const *templates,
                              uintptr_t n_templates, bool on_device, SketchCollection **out) {
    if (out)
        for (uintptr_t m = 0; m < n_templates; m++) out[m] = nullptr;
    landingpad_void([&]() {
        nonnull(out, "out");
        if (n_templates) nonnull(templates, "templates");
        if (n_seqs) { nonnull(offsets, "offsets"); }
        if (n_templates < 1 || n_templates > 6) smb200::throw_internal("sketch_collections takes 1 to 6 templates");
        std::vector<smb200::SketchParams> ps(n_templates);
        {
            GuardN lk;
            for (uintptr_t m = 0; m < n_templates; m++) lk.add(mh(templates[m])->mu);
            lk.lock();
            for (uintptr_t m = 0; m < n_templates; m++) {
                const MH *t = mh(templates[m]);
                if (t->track_abundance())
                    smb200::throw_internal("a sketch collection holds no abundances: a template that tracks abundance is refused");
                ps[m] = {t->num, t->ksize, t->is_protein, t->seed, t->max_hash};
            }
        }
        std::vector<std::unique_ptr<COLL>> cs =
            smb200::sketch_collections(reinterpret_cast<const uint8_t *>(buf), offsets, n_seqs, ps, on_device);
        for (uintptr_t m = 0; m < n_templates; m++) out[m] = reinterpret_cast<SketchCollection *>(cs[m].release());
    });
}
uint64_t smgpu_collection_len(SketchCollection *c) {
    return landingpad<uint64_t>([&]() { COLL *cc = coll(c); Guard lk(cc->mu); return cc->dirty ? (uint64_t)cc->h_nums.size() : cc->n_rows; });
}
uint64_t smgpu_collection_copy(SketchCollection *c, uint64_t *hashes, uint64_t *offsets) {
    return landingpad<uint64_t>([&]() -> uint64_t {
        COLL *cc = coll(c);
        Guard lk(cc->mu);
        cc->finalize();
        smb200::Context &ctx = smb200::Context::get();
        if (offsets) std::copy(cc->h_offsets.begin(), cc->h_offsets.begin() + cc->n_rows + 1, offsets);
        if (hashes && cc->n_hashes) {
            SM_CUDA(cudaMemcpyAsync(hashes, cc->d_hashes.p, cc->n_hashes * 8, cudaMemcpyDeviceToHost, ctx.stream));
            ctx.sync();
        }
        return cc->n_hashes;
    });
}
uint64_t smgpu_collection_csr(SketchCollection *c, const uint64_t **hashes_dev, const uint64_t **offsets_dev) {
    return landingpad<uint64_t>([&]() {
        COLL *cc = coll(c);
        Guard lk(cc->mu);
        cc->finalize();
        if (hashes_dev) *hashes_dev = cc->d_hashes.as<uint64_t>();
        if (offsets_dev) *offsets_dev = cc->d_offsets.as<uint64_t>();
        return cc->n_hashes;
    });
}
void smgpu_compare_matrix(SketchCollection *rows, uint64_t r0, uint64_t nr, SketchCollection *cols, uint64_t c0, uint64_t nc,
                          int32_t mode, uint32_t *common, uint32_t *size, double *ratio, uint64_t ld, bool out_on_device) {
    landingpad_void([&]() {
        if (mode != 0 && mode != 1) smb200::throw_internal("mode must be 0 (compare) or 1 (containment)");
        COLL *r = coll(rows), *c = coll(cols);
        Guard lk(r->mu, c->mu);
        smb200::compare_matrix(*r, r0, nr, *c, c0, nc, mode, common, size, ratio, ld, out_on_device);
    });
}
uint64_t smgpu_scaffold_pairs(SketchCollection *c, uint64_t *pairs_first, uint64_t *pairs_second) {
    return landingpad<uint64_t>([&]() {
        nonnull(pairs_first, "pairs_first");
        nonnull(pairs_second, "pairs_second");
        COLL *cc = coll(c);
        Guard lk(cc->mu);
        return smb200::scaffold_pairs(*cc, pairs_first, pairs_second);
    });
}
void smgpu_fuse_multi_k(bool on) { smb200::g_fuse_multi_k = on; }
void smgpu_find_path(int32_t path) { smb200::g_find_path = (path >= 0 && path <= 3) ? path : 0; }
void smgpu_compare_path(int32_t path) { smb200::g_compare_path = (path >= 1 && path <= 2) ? path : 0; }
uint64_t smgpu_linear_find(SketchCollection *index, SketchCollection *queries, int32_t mode, double threshold,
                           uint64_t *hit_offsets, uint64_t *hits, uint64_t hits_cap) {
    return landingpad<uint64_t>([&]() {
        if (mode != 0 && mode != 1) smb200::throw_internal("mode must be 0 (similarity) or 1 (containment)");
        COLL *ix = coll(index), *q = coll(queries);
        Guard lk(ix->mu, q->mu);
        return smb200::linear_find(*ix, *q, mode, threshold, hit_offsets, hits, hits_cap);
    });
}


// ---- multi-GPU: one process per GPU, NCCL inside the library (comm.cu) -----------------------------------
void smgpu_comm_unique_id(uint8_t *id128) {
    landingpad_void([&]() { nonnull(id128, "id128"); smb200::comm_unique_id(id128); });
}
void smgpu_comm_init(const uint8_t *id128, int32_t rank, int32_t world) {
    landingpad_void([&]() { nonnull(id128, "id128"); smb200::comm_init(id128, rank, world); });
}
void smgpu_comm_destroy(void) { landingpad_void([&]() { smb200::comm_destroy(); }); }
int32_t smgpu_comm_rank(void) { return smb200::comm_rank(); }
int32_t smgpu_comm_world(void) { return smb200::comm_world(); }
int32_t smgpu_comm_nccl_version(void) { return landingpad<int32_t>([&]() { return (int32_t)smb200::comm_nccl_version(); }); }
SketchCollection *smgpu_collection_allgather(SketchCollection *local) {
    return landingpad<SketchCollection *>([&]() {
        COLL *l = coll(local);
        Guard lk(l->mu);
        return reinterpret_cast<SketchCollection *>(smb200::collection_allgather(*l));
    });
}
SketchCollection *smgpu_compare_matrix_allgather(SketchCollection *local, int32_t mode, uint32_t *common, uint32_t *size, double *ratio,
                                                 uint64_t ld, bool out_on_device) {
    return landingpad<SketchCollection *>([&]() {
        if (mode != 0 && mode != 1) smb200::throw_internal("mode must be 0 (compare) or 1 (containment)");
        COLL *l = coll(local);
        Guard lk(l->mu);
        return reinterpret_cast<SketchCollection *>(smb200::compare_matrix_allgather(*l, mode, common, size, ratio, ld, out_on_device));
    });
}
void smgpu_comm_allmerge(KmerMinHash *ptr) {
    landingpad_void([&]() { MH *m = mh(ptr); Guard lk(m->mu); smb200::comm_allmerge(*m); });
}
uint64_t smgpu_linear_find_sharded(SketchCollection *index_part, SketchCollection *queries, int32_t mode, double threshold,
                                   uint64_t *hit_offsets, uint64_t *hits, uint64_t hits_cap) {
    return landingpad<uint64_t>([&]() {
        if (mode != 0 && mode != 1) smb200::throw_internal("mode must be 0 (similarity) or 1 (containment)");
        COLL *ix = coll(index_part), *q = coll(queries);
        Guard lk(ix->mu, q->mu);
        return smb200::linear_find_sharded(*ix, *q, mode, threshold, hit_offsets, hits, hits_cap);
    });
}

// ---- Nodegraph / SBT (src/index/nodegraph.rs, src/index/sbt.rs) ---------------------------------------
Nodegraph *smgpu_nodegraph_new(const uint64_t *tablesizes, uintptr_t n_tables, uint64_t ksize) {
    return landingpad<Nodegraph *>([&]() {
        if (n_tables) nonnull(tablesizes, "tablesizes");
        return reinterpret_cast<Nodegraph *>(new NG(tablesizes, n_tables, ksize));
    });
}
void smgpu_nodegraph_free(Nodegraph *ng) {
    landingpad_void([&]() { delete reinterpret_cast<NG *>(ng); });
}
Nodegraph *smgpu_nodegraph_from_buffer(const uint8_t *data, uintptr_t len) {
    return landingpad<Nodegraph *>([&]() {
        nonnull(data, "data");
        return reinterpret_cast<Nodegraph *>(NG::from_buffer(data, len));
    });
}
uintptr_t smgpu_nodegraph_save(Nodegraph *ng, uint8_t *out, uintptr_t cap) {
    return landingpad<uintptr_t>([&]() -> uintptr_t { NG *g = ngp(ng); Guard lk(g->mu); return g->save(out, out ? cap : 0); });
}
uint64_t smgpu_nodegraph_count_many(Nodegraph *ng, const uint64_t *hashes, uint64_t n, uint8_t *is_new, bool on_device) {
    return landingpad<uint64_t>([&]() -> uint64_t {
        if (n) nonnull(hashes, "hashes");
        NG *g = ngp(ng);
        Guard lk(g->mu);
        return g->count_many(hashes, n, is_new, on_device);
    });
}
uint64_t smgpu_nodegraph_get_many(Nodegraph *ng, const uint64_t *hashes, uint64_t n, uint8_t *present, bool on_device) {
    return landingpad<uint64_t>([&]() -> uint64_t {
        if (n) nonnull(hashes, "hashes");
        NG *g = ngp(ng);
        Guard lk(g->mu);
        return g->get_many(hashes, n, present, on_device);
    });
}
uint64_t smgpu_nodegraph_matches(Nodegraph *ng, KmerMinHash *ptr) {
    return landingpad<uint64_t>([&]() -> uint64_t {
        size_t n = 0;
        NG *g = ngp(ng);
        MH *m = mh(ptr);
        Guard lk(g->mu, m->mu);
        const uint64_t *dm = m->device_mins(&n);
        return g->get_many(dm, n, nullptr, true);
    });
}
void smgpu_nodegraph_update(Nodegraph *ng, Nodegraph *other) {
    landingpad_void([&]() { NG *a = ngp(ng), *b = ngp(other); Guard lk(a->mu, b->mu); a->update(*b); });
}
double smgpu_nodegraph_similarity(Nodegraph *ng, Nodegraph *other) {
    return landingpad<double>([&]() { NG *a = ngp(ng), *b = ngp(other); Guard lk(a->mu, b->mu); return a->similarity(*b); });
}
double smgpu_nodegraph_containment(Nodegraph *ng, Nodegraph *other) {
    return landingpad<double>([&]() { NG *a = ngp(ng), *b = ngp(other); Guard lk(a->mu, b->mu); return a->containment(*b); });
}
uintptr_t smgpu_nodegraph_tablesizes(Nodegraph *ng, uint64_t *out, uintptr_t cap) {
    return landingpad<uintptr_t>([&]() -> uintptr_t {
        NG *g = ngp(ng);
        for (size_t t = 0; out && t < g->tables.size() && t < cap; t++) out[t] = g->tables[t].len;
        return g->tables.size();
    });
}
uint64_t smgpu_nodegraph_ksize(Nodegraph *ng) { return landingpad<uint64_t>([&]() { return ngp(ng)->ksize; }); }
uint64_t smgpu_nodegraph_n_occupied_bins(Nodegraph *ng) { return landingpad<uint64_t>([&]() { NG *g = ngp(ng); Guard lk(g->mu); return g->occupied_bins; }); }
uint64_t smgpu_nodegraph_unique_kmers(Nodegraph *ng) { return landingpad<uint64_t>([&]() { NG *g = ngp(ng); Guard lk(g->mu); return g->unique_kmers; }); }
uint64_t smgpu_sbt_find(uint32_t d, const uint64_t *node_positions, Nodegraph *const *nodes, const uint64_t *min_n_below,
                        uint64_t n_nodes, const uint64_t *leaf_positions, SketchCollection *leaves, SketchCollection *queries,
                        int32_t mode, double threshold, uint64_t *hit_offsets, uint64_t *hits, uint64_t hits_cap) {
    return landingpad<uint64_t>([&]() -> uint64_t {
        if (mode != 0 && mode != 1) smb200::throw_internal("mode must be 0 (similarity) or 1 (containment)");
        if (d == 0) smb200::throw_internal("d must be at least 1");
        if (n_nodes) { nonnull(node_positions, "node_positions"); nonnull(nodes, "nodes"); nonnull(min_n_below, "min_n_below"); }
        for (uint64_t i = 0; i < n_nodes; i++) ngp(nodes[i]);
        COLL *l = coll(leaves);
        GuardN lk;
        lk.add(l->mu);
        lk.add(coll(queries)->mu);
        for (uint64_t i = 0; i < n_nodes; i++) lk.add(ngp(nodes[i])->mu);
        lk.lock();
        l->finalize();
        if (l->n_rows) nonnull(leaf_positions, "leaf_positions");
        return smb200::sbt_find(d, node_positions, reinterpret_cast<NG *const *>(nodes), min_n_below, n_nodes, leaf_positions, *l,
                                *coll(queries), mode, threshold, hit_offsets, hits, hits_cap);
    });
}

}  // extern "C"
