/*
 * oracle.c -- CPU restatement of sourmash-rust's sketch-and-compare path.
 *
 * TEST INFRASTRUCTURE ONLY.  Nothing under sourmash_rust_b200/ may include,
 * link or call this file; only tests/, __graft_entry__.smoke() and bench.py's
 * cpu_baseline / --impl reference legs use it, as the checker / CPU baseline.
 *
 * Every function cites the reference file:line (relative to /root/reference)
 * whose behaviour it restates.  The structure deliberately follows the
 * reference (whole-sequence uppercase copy, per-window validity scan,
 * allocating reverse complement, byte-wise lexicographic min, binary-search
 * insert, three-pass compare) because it doubles as the CPU baseline.
 *
 * Parity pins (tests/test_oracle.py): tests/test.rs:5 (hash KAT),
 * tests/minhash.rs:19-83 (merge KAT, compare), src/index/sbt.rs:543-588 hit
 * counts over the .sbt.v5 fixtures, md5sum of all 11 sorted fixture sketches,
 * and the SMHasher verification value 0x6384BA69 for the 16-byte body loop
 * that no reference test reaches ("parity unpinned" by the reference itself).
 *
 * MurmurHash3 x64_128 is third-party to the reference (crate `murmurhash3`
 * ~0.0.5, Cargo.toml:49; called at src/lib.rs:33-35).  It is restated here from
 * the published algorithm (Austin Appleby, public domain); the crate seeds
 * h1 = h2 = seed as a full u64.
 */
#include <stdint.h>
#include <stdlib.h>
#include <string.h>
#include <stdio.h>
#include <math.h>

/* ------------------------------------------------------------------ */
/* growable u64 / byte vectors                                          */
/* ------------------------------------------------------------------ */
typedef struct {
    uint64_t *p;
    size_t len, cap;
} vec64;

static void v_reserve(vec64 *v, size_t n) {
    if (n <= v->cap) return;
    size_t c = v->cap ? v->cap : 16;
    while (c < n) c *= 2;
    v->p = (uint64_t *)realloc(v->p, c * sizeof(uint64_t));
    v->cap = c;
}
static void v_push(vec64 *v, uint64_t x) {
    v_reserve(v, v->len + 1);
    v->p[v->len++] = x;
}
static void v_insert(vec64 *v, size_t pos, uint64_t x) {
    v_reserve(v, v->len + 1);
    memmove(v->p + pos + 1, v->p + pos, (v->len - pos) * sizeof(uint64_t));
    v->p[pos] = x;
    v->len++;
}
static void v_free(vec64 *v) {
    free(v->p);
    v->p = NULL;
    v->len = v->cap = 0;
}
static void v_copy(vec64 *dst, const vec64 *src) {
    dst->len = 0;
    v_reserve(dst, src->len);
    if (src->len) memcpy(dst->p, src->p, src->len * sizeof(uint64_t));
    dst->len = src->len;
}

typedef struct {
    char *p;
    size_t len, cap;
} sbuf;
static void s_reserve(sbuf *s, size_t n) {
    if (n <= s->cap) return;
    size_t c = s->cap ? s->cap : 256;
    while (c < n) c *= 2;
    s->p = (char *)realloc(s->p, c);
    s->cap = c;
}
static void s_put(sbuf *s, const char *d, size_t n) {
    s_reserve(s, s->len + n + 1);
    memcpy(s->p + s->len, d, n);
    s->len += n;
    s->p[s->len] = 0;
}
static void s_puts(sbuf *s, const char *d) { s_put(s, d, strlen(d)); }
static void s_putu(sbuf *s, uint64_t x) {
    char t[24];
    int n = snprintf(t, sizeof t, "%llu", (unsigned long long)x);
    s_put(s, t, (size_t)n);
}

/* ------------------------------------------------------------------ */
/* MurmurHash3 x64_128 (third-party boundary; lib.rs:29,33-35)          */
/* ------------------------------------------------------------------ */
static inline uint64_t rotl64(uint64_t x, int r) { return (x << r) | (x >> (64 - r)); }
static inline uint64_t fmix64(uint64_t k) {
    k ^= k >> 33;
    k *= 0xff51afd7ed558ccdULL;
    k ^= k >> 33;
    k *= 0xc4ceb9fe1a85ec53ULL;
    k ^= k >> 33;
    return k;
}

void orc_murmur3_x64_128(const uint8_t *data, size_t len, uint64_t seed, uint64_t out[2]) {
    const uint64_t c1 = 0x87c37b91114253d5ULL, c2 = 0x4cf5ad432745937fULL;
    uint64_t h1 = seed, h2 = seed;
    size_t nblocks = len / 16;
    for (size_t i = 0; i < nblocks; i++) {
        uint64_t k1, k2;
        memcpy(&k1, data + 16 * i, 8);     /* little-endian block read */
        memcpy(&k2, data + 16 * i + 8, 8);
        k1 *= c1; k1 = rotl64(k1, 31); k1 *= c2; h1 ^= k1;
        h1 = rotl64(h1, 27); h1 += h2; h1 = h1 * 5 + 0x52dce729;
        k2 *= c2; k2 = rotl64(k2, 33); k2 *= c1; h2 ^= k2;
        h2 = rotl64(h2, 31); h2 += h1; h2 = h2 * 5 + 0x38495ab5;
    }
    const uint8_t *tail = data + nblocks * 16;
    uint64_t k1 = 0, k2 = 0;
    switch (len & 15) {
    case 15: k2 ^= (uint64_t)tail[14] << 48; /* fallthrough */
    case 14: k2 ^= (uint64_t)tail[13] << 40; /* fallthrough */
    case 13: k2 ^= (uint64_t)tail[12] << 32; /* fallthrough */
    case 12: k2 ^= (uint64_t)tail[11] << 24; /* fallthrough */
    case 11: k2 ^= (uint64_t)tail[10] << 16; /* fallthrough */
    case 10: k2 ^= (uint64_t)tail[9] << 8;   /* fallthrough */
    case 9:  k2 ^= (uint64_t)tail[8];
             k2 *= c2; k2 = rotl64(k2, 33); k2 *= c1; h2 ^= k2; /* fallthrough */
    case 8:  k1 ^= (uint64_t)tail[7] << 56;  /* fallthrough */
    case 7:  k1 ^= (uint64_t)tail[6] << 48;  /* fallthrough */
    case 6:  k1 ^= (uint64_t)tail[5] << 40;  /* fallthrough */
    case 5:  k1 ^= (uint64_t)tail[4] << 32;  /* fallthrough */
    case 4:  k1 ^= (uint64_t)tail[3] << 24;  /* fallthrough */
    case 3:  k1 ^= (uint64_t)tail[2] << 16;  /* fallthrough */
    case 2:  k1 ^= (uint64_t)tail[1] << 8;   /* fallthrough */
    case 1:  k1 ^= (uint64_t)tail[0];
             k1 *= c1; k1 = rotl64(k1, 31); k1 *= c2; h1 ^= k1;
    }
    h1 ^= (uint64_t)len; h2 ^= (uint64_t)len;
    h1 += h2; h2 += h1;
    h1 = fmix64(h1); h2 = fmix64(h2);
    h1 += h2; h2 += h1;
    out[0] = h1; out[1] = h2;
}

/* lib.rs:33-35  _hash_murmur: first u64 of the pair */
uint64_t orc_hash_murmur(const uint8_t *kmer, size_t len, uint64_t seed) {
    uint64_t o[2];
    orc_murmur3_x64_128(kmer, len, seed, o);
    return o[0];
}

/* SMHasher VerificationTest for MurmurHash3_x64_128 (expected 0x6384BA69):
 * keys {0},{0,1},... hashed with seed 256-i; hash the 256 results with seed 0;
 * first 4 bytes little-endian.  Pins the 16-byte body loop. */
uint32_t orc_smhasher_verification(void) {
    uint8_t key[256], hashes[256 * 16];
    uint64_t o[2];
    for (int i = 0; i < 256; i++) {
        key[i] = (uint8_t)i;
        orc_murmur3_x64_128(key, (size_t)i, (uint64_t)(uint32_t)(256 - i), o);
        memcpy(hashes + 16 * i, o, 16);
    }
    orc_murmur3_x64_128(hashes, sizeof hashes, 0, o);
    return (uint32_t)(o[0] & 0xffffffffu);
}

/* ------------------------------------------------------------------ */
/* KmerMinHash (lib.rs:37-46)                                           */
/* ------------------------------------------------------------------ */
typedef struct {
    uint32_t num, ksize;
    int is_protein;
    uint64_t seed, max_hash;
    vec64 mins;
    int has_abunds; /* abunds: Option<Vec<u64>> */
    vec64 abunds;
} OrcMinHash;

enum {
    ORC_OK = 0,
    ORC_MISMATCH_KSIZES = 101,
    ORC_MISMATCH_DNAPROT = 102,
    ORC_MISMATCH_MAXHASH = 103,
    ORC_MISMATCH_SEED = 104,
    ORC_INVALID_DNA = 1101,
    ORC_UNSUPPORTED = 2
};

/* lib.rs:142-174 */
OrcMinHash *orc_mh_new(uint32_t num, uint32_t ksize, int is_protein, uint64_t seed,
                       uint64_t max_hash, int track_abundance) {
    OrcMinHash *mh = (OrcMinHash *)calloc(1, sizeof *mh);
    mh->num = num; mh->ksize = ksize; mh->is_protein = is_protein;
    mh->seed = seed; mh->max_hash = max_hash;
    v_reserve(&mh->mins, num > 0 ? num : 1000);
    mh->has_abunds = track_abundance ? 1 : 0;
    return mh;
}
void orc_mh_free(OrcMinHash *mh) {
    if (!mh) return;
    v_free(&mh->mins); v_free(&mh->abunds); free(mh);
}
OrcMinHash *orc_mh_clone(const OrcMinHash *o) {
    OrcMinHash *mh = orc_mh_new(o->num, o->ksize, o->is_protein, o->seed, o->max_hash, o->has_abunds);
    v_copy(&mh->mins, &o->mins);
    v_copy(&mh->abunds, &o->abunds);
    return mh;
}
size_t orc_mh_size(const OrcMinHash *mh) { return mh->mins.len; }
const uint64_t *orc_mh_mins(const OrcMinHash *mh) { return mh->mins.p; }
size_t orc_mh_abunds_size(const OrcMinHash *mh) { return mh->has_abunds ? mh->abunds.len : 0; }
const uint64_t *orc_mh_abunds(const OrcMinHash *mh) { return mh->has_abunds ? mh->abunds.p : NULL; }
int orc_mh_track_abundance(const OrcMinHash *mh) { return mh->has_abunds; }
uint32_t orc_mh_num(const OrcMinHash *mh) { return mh->num; }
/* ffi.rs:143-150, 179-188: raw appends */
void orc_mh_mins_push(OrcMinHash *mh, uint64_t v) { v_push(&mh->mins, v); }
void orc_mh_abunds_push(OrcMinHash *mh, uint64_t v) { if (mh->has_abunds) v_push(&mh->abunds, v); }

/* lib.rs:176-190 -- order of the checks matters */
int orc_mh_check_compatible(const OrcMinHash *a, const OrcMinHash *b) {
    if (a->ksize != b->ksize) return ORC_MISMATCH_KSIZES;
    if (a->is_protein != b->is_protein) return ORC_MISMATCH_DNAPROT;
    if (a->max_hash != b->max_hash) return ORC_MISMATCH_MAXHASH;
    if (a->seed != b->seed) return ORC_MISMATCH_SEED;
    return ORC_OK;
}

/* slice::binary_search on a sorted slice: returns insertion point, sets *found.
 * (When duplicates exist Rust may return any match; mins are distinct here.) */
static size_t bsearch64(const uint64_t *p, size_t n, uint64_t x, int *found) {
    size_t lo = 0, hi = n;
    *found = 0;
    while (lo < hi) {
        size_t mid = lo + (hi - lo) / 2;
        if (p[mid] == x) { *found = 1; return mid; }
        if (p[mid] < x) lo = mid + 1; else hi = mid;
    }
    return lo;
}

/* lib.rs:192-245 -- the sketch state machine, restated branch for branch */
void orc_mh_add_hash(OrcMinHash *mh, uint64_t hash) {
    uint64_t current_max = mh->mins.len ? mh->mins.p[mh->mins.len - 1] : UINT64_MAX;
    if (hash <= mh->max_hash || mh->max_hash == 0) {
        if (mh->mins.len == 0) {
            v_push(&mh->mins, hash);
            if (mh->has_abunds) v_push(&mh->abunds, 1);
            return;
        } else if (hash <= mh->max_hash || current_max > hash ||
                   (uint32_t)mh->mins.len < mh->num) {
            int found;
            size_t pos = bsearch64(mh->mins.p, mh->mins.len, hash, &found);
            if (pos == mh->mins.len) {
                v_push(&mh->mins, hash);
                if (mh->has_abunds) v_push(&mh->abunds, 1);
            } else if (mh->mins.p[pos] != hash) {
                v_insert(&mh->mins, pos, hash);
                if (mh->has_abunds) v_insert(&mh->abunds, pos, 1);
                if (mh->num != 0 && mh->mins.len > (size_t)mh->num) {
                    mh->mins.len--;
                    if (mh->has_abunds) mh->abunds.len--;
                }
            } else if (mh->has_abunds) {
                mh->abunds.p[pos] += 1;
            }
        }
    }
}

/* lib.rs:247-250 */
void orc_mh_add_word(OrcMinHash *mh, const uint8_t *word, size_t len) {
    orc_mh_add_hash(mh, orc_hash_murmur(word, len, mh->seed));
}

/* lib.rs:795-804 */
static int checkdna(const uint8_t *s, size_t n) {
    for (size_t i = 0; i < n; i++) {
        switch (s[i]) {
        case 'A': case 'C': case 'G': case 'T':
        case 'a': case 'c': case 'g': case 't': break;
        default: return 0;
        }
    }
    return 1;
}

/* lib.rs:677-689 -- allocates a fresh buffer per call, like the reference */
static uint8_t *revcomp_alloc(const uint8_t *s, size_t n) {
    uint8_t *rc = (uint8_t *)malloc(n ? n : 1);
    for (size_t i = 0; i < n; i++) {
        uint8_t c = s[n - 1 - i], o;
        switch (c) {
        case 'A': case 'a': o = 'T'; break;
        case 'T': case 't': o = 'A'; break;
        case 'C': case 'c': o = 'G'; break;
        case 'G': case 'g': o = 'C'; break;
        default: o = c;
        }
        rc[i] = o;
    }
    return rc;
}

/* CODONTABLE (lib.rs:691-763): the standard genetic code, stops as '*'; anything that is not three
 * upper-case ACGT letters has no entry */
static int codon_code(uint8_t c) { return c == 'A' ? 0 : c == 'C' ? 1 : c == 'G' ? 2 : c == 'T' ? 3 : -1; }
static uint8_t codon_lookup(const uint8_t *c3) {
    static const char table[65] = "KNKNTTTTRSRSIIMIQHQHPPPPRRRRLLLLEDEDAAAAGGGGVVVV*Y*YSSSS*CWCLFLF"; /* index 16a+4b+c, A0 C1 G2 T3 */
    const int a = codon_code(c3[0]), b = codon_code(c3[1]), c = codon_code(c3[2]);
    if (a < 0 || b < 0 || c < 0) return 0;
    return (uint8_t)table[16 * a + 4 * b + c];
}
/* to_aa (lib.rs:776-793): chunks of 3, an incomplete last chunk ends it, unknown codons are skipped */
static size_t to_aa(const uint8_t *s, size_t n, uint8_t *out) {
    size_t m = 0;
    for (size_t i = 0; i + 3 <= n; i += 3) {
        const uint8_t aa = codon_lookup(s + i);
        if (aa) out[m++] = aa;
    }
    return m;
}

/* lib.rs:252-305.  DNA arm: on an invalid k-mer with !force returns ORC_INVALID_DNA and copies the
 * offending (uppercased) k-mer into badkmer (ksize bytes + NUL) -- k-mers before it stay added
 * (partial mutation).  Protein arm (lib.rs:275-302): the three forward frames and the three frames
 * of the reverse complement are translated and every window of ksize/3 residues is hashed; no
 * validity check, `force` is not consulted. */
int orc_mh_add_sequence(OrcMinHash *mh, const uint8_t *seq, size_t len, int force, char *badkmer) {
    uint8_t *sequence = (uint8_t *)malloc(len ? len : 1);
    for (size_t i = 0; i < len; i++) {
        uint8_t c = seq[i];
        sequence[i] = (c >= 'a' && c <= 'z') ? (uint8_t)(c - 32) : c; /* lib.rs:253-256 */
    }
    int rc_code = ORC_OK;
    size_t k = mh->ksize;
    if (mh->is_protein) {
        if (len >= k) {
            const size_t aa_k = k / 3;
            if (aa_k == 0) { free(sequence); return ORC_UNSUPPORTED; } /* slice::windows(0) panics */
            uint8_t *rc = revcomp_alloc(sequence, len);
            uint8_t *aa = (uint8_t *)malloc(len / 3 + 1);
            for (size_t i = 0; i < 3; i++) {
                const size_t sub = len >= i ? len - i : 0;
                size_t m = to_aa(sequence + (len >= i ? i : len), sub, aa);
                for (size_t w = 0; w + aa_k <= m; w++) orc_mh_add_word(mh, aa + w, aa_k);
                m = to_aa(rc + (len >= i ? i : len), sub, aa);
                for (size_t w = 0; w + aa_k <= m; w++) orc_mh_add_word(mh, aa + w, aa_k);
            }
            free(aa);
            free(rc);
        }
        free(sequence);
        return ORC_OK;
    }
    if (len >= k && k > 0) {
        for (size_t i = 0; i + k <= len; i++) {
            const uint8_t *kmer = sequence + i;
            if (checkdna(kmer, k)) {
                uint8_t *rc = revcomp_alloc(kmer, k);
                if (memcmp(kmer, rc, k) < 0) orc_mh_add_word(mh, kmer, k);
                else orc_mh_add_word(mh, rc, k);
                free(rc);
            } else if (!force) {
                if (badkmer) { memcpy(badkmer, kmer, k); badkmer[k] = 0; }
                rc_code = ORC_INVALID_DNA;
                break;
            }
        }
    }
    free(sequence);
    return rc_code;
}

/* lib.rs:405-417 */
void orc_mh_add_many(OrcMinHash *mh, const uint64_t *h, size_t n) {
    for (size_t i = 0; i < n; i++) orc_mh_add_hash(mh, h[i]);
}
void orc_mh_add_from(OrcMinHash *mh, const OrcMinHash *o) { orc_mh_add_many(mh, o->mins.p, o->mins.len); }

/* lib.rs:307-403 -- including the abundance quirks: abunds is forced to
 * Some(..) afterwards, is not truncated with mins, and goes out of step when
 * only one side tracks abundance. */
int orc_mh_merge(OrcMinHash *self, const OrcMinHash *other) {
    int e = orc_mh_check_compatible(self, other);
    if (e) return e;
    vec64 merged = {0}, mab = {0};
    v_reserve(&merged, self->mins.len + other->mins.len);
    v_reserve(&mab, self->mins.len + other->mins.len);
    size_t si = 0, oi = 0, sa = 0, oa = 0;
    const int has_sa = self->has_abunds, has_oa = other->has_abunds;
    const size_t sn = self->mins.len, on = other->mins.len;
    const size_t san = self->abunds.len, oan = other->abunds.len;
    int sv_some = si < sn; uint64_t sv = sv_some ? self->mins.p[si++] : 0;
    int ov_some = oi < on; uint64_t ov = ov_some ? other->mins.p[oi++] : 0;
    while (sv_some) {
        if (!ov_some) {
            v_push(&merged, sv);
            while (si < sn) v_push(&merged, self->mins.p[si++]);
            if (has_sa) while (sa < san) v_push(&mab, self->abunds.p[sa++]);
            break;
        } else if (ov < sv) {
            v_push(&merged, ov);
            ov_some = oi < on; if (ov_some) ov = other->mins.p[oi++];
            if (has_oa && oa < oan) v_push(&mab, other->abunds.p[oa++]);
        } else if (ov == sv) {
            v_push(&merged, ov);
            ov_some = oi < on; if (ov_some) ov = other->mins.p[oi++];
            sv_some = si < sn; if (sv_some) sv = self->mins.p[si++];
            if (has_oa && oa < oan) {
                uint64_t v = other->abunds.p[oa++];
                if (has_sa && sa < san) v_push(&mab, v + self->abunds.p[sa++]);
            }
        } else {
            v_push(&merged, sv);
            sv_some = si < sn; if (sv_some) sv = self->mins.p[si++];
            if (has_sa && sa < san) v_push(&mab, self->abunds.p[sa++]);
        }
    }
    if (ov_some) v_push(&merged, ov);
    while (oi < on) v_push(&merged, other->mins.p[oi++]);
    if (has_oa) while (oa < oan) v_push(&mab, other->abunds.p[oa++]);

    if (!(merged.len < (size_t)self->num || self->num == 0)) merged.len = self->num; /* lib.rs:391-401 */
    v_free(&self->mins); v_free(&self->abunds);
    self->mins = merged;
    self->abunds = mab;
    self->has_abunds = 1; /* lib.rs:393,400 */
    return ORC_OK;
}

/* lib.rs:515-544 -- two-pointer intersection; writes matches to out if non-NULL */
static size_t intersection_walk(const uint64_t *l, size_t ln, const uint64_t *r, size_t rn, vec64 *out) {
    size_t i = 0, j = 0, c = 0;
    while (i < ln && j < rn) {
        if (l[i] < r[j]) i++;
        else if (l[i] > r[j]) j++;
        else { if (out) v_push(out, l[i]); c++; i++; j++; }
    }
    return c;
}

/* lib.rs:428-436 */
int orc_mh_count_common(const OrcMinHash *a, const OrcMinHash *b, uint64_t *common) {
    int e = orc_mh_check_compatible(a, b);
    *common = 0;
    if (e) return e;
    *common = intersection_walk(a->mins.p, a->mins.len, b->mins.p, b->mins.len, NULL);
    return ORC_OK;
}

/* lib.rs:470-499 (and :438-468 when out_common != NULL) */
int orc_mh_intersection_size(const OrcMinHash *a, const OrcMinHash *b, uint64_t *common, uint64_t *size) {
    int e = orc_mh_check_compatible(a, b);
    *common = 0; *size = 0;
    if (e) return e;
    OrcMinHash *comb = orc_mh_new(a->num, a->ksize, a->is_protein, a->seed, a->max_hash, a->has_abunds);
    orc_mh_merge(comb, a);
    orc_mh_merge(comb, b);
    vec64 i1 = {0};
    intersection_walk(a->mins.p, a->mins.len, b->mins.p, b->mins.len, &i1);
    *common = intersection_walk(i1.p, i1.len, comb->mins.p, comb->mins.len, NULL);
    *size = comb->mins.len;
    v_free(&i1);
    orc_mh_free(comb);
    return ORC_OK;
}

/* lib.rs:438-468: the common hashes themselves (those of A n B also in combined) and |combined|.
 * out receives at most cap of them; *n_common the number there are. */
int orc_mh_intersection(const OrcMinHash *a, const OrcMinHash *b, uint64_t *out, size_t cap, uint64_t *n_common, uint64_t *size) {
    int e = orc_mh_check_compatible(a, b);
    *n_common = 0; *size = 0;
    if (e) return e;
    OrcMinHash *comb = orc_mh_new(a->num, a->ksize, a->is_protein, a->seed, a->max_hash, a->has_abunds);
    orc_mh_merge(comb, a);
    orc_mh_merge(comb, b);
    vec64 i1 = {0}, common = {0};
    intersection_walk(a->mins.p, a->mins.len, b->mins.p, b->mins.len, &i1);
    intersection_walk(i1.p, i1.len, comb->mins.p, comb->mins.len, &common);
    *n_common = common.len;
    *size = comb->mins.len;
    for (size_t i = 0; i < common.len && i < cap; i++) out[i] = common.p[i];
    v_free(&i1); v_free(&common);
    orc_mh_free(comb);
    return ORC_OK;
}

/* lib.rs:501-508 */
int orc_mh_compare(const OrcMinHash *a, const OrcMinHash *b, double *out) {
    uint64_t common, size;
    *out = 0.0;
    int e = orc_mh_intersection_size(a, b, &common, &size);
    if (e) return e;
    *out = (double)common / (double)(size > 1 ? size : 1);
    return ORC_OK;
}

/* index.rs:131-144 (similarity) and :146-160 (containment: |node∩query|/|node|) */
double orc_leaf_similarity(const OrcMinHash *node, const OrcMinHash *query) {
    double d = 0.0;
    orc_mh_compare(node, query, &d);
    return d;
}
double orc_leaf_containment(const OrcMinHash *node, const OrcMinHash *query) {
    uint64_t c = 0;
    orc_mh_count_common(node, query, &c);
    return (double)c / (double)node->mins.len; /* 0/0 -> NaN, never > thr */
}

/* linear.rs:25-45 with search.rs:3-9: ordered scan, strict '>' threshold.
 * mode 0 = search_minhashes, 1 = search_minhashes_containment. Returns #hits,
 * hit indices (insertion order) in hits[]. */
size_t orc_linear_find(OrcMinHash *const *leaves, size_t n, const OrcMinHash *query, int mode,
                       double threshold, uint64_t *hits) {
    size_t nh = 0;
    for (size_t i = 0; i < n; i++) {
        double v = mode ? orc_leaf_containment(leaves[i], query) : orc_leaf_similarity(leaves[i], query);
        if (v > threshold) hits[nh++] = i;
    }
    return nh;
}

/* batch helpers for the tests / CPU baseline (plain loops over the above) */
void orc_compare_matrix(OrcMinHash *const *rows, size_t nr, OrcMinHash *const *cols, size_t nc,
                        uint32_t *common, uint32_t *size, double *jaccard) {
    for (size_t i = 0; i < nr; i++)
        for (size_t j = 0; j < nc; j++) {
            uint64_t c, s;
            orc_mh_intersection_size(rows[i], cols[j], &c, &s);
            if (common) common[i * nc + j] = (uint32_t)c;
            if (size) size[i * nc + j] = (uint32_t)s;
            if (jaccard) jaccard[i * nc + j] = (double)c / (double)(s > 1 ? s : 1);
        }
}
void orc_count_common_matrix(OrcMinHash *const *rows, size_t nr, OrcMinHash *const *cols, size_t nc,
                             uint32_t *common) {
    for (size_t i = 0; i < nr; i++)
        for (size_t j = 0; j < nc; j++) {
            uint64_t c;
            orc_mh_count_common(rows[i], cols[j], &c);
            common[i * nc + j] = (uint32_t)c;
        }
}
/* scaffold's leaf-pairing pass (src/index/sbt.rs:356-381): pop the LAST dataset, find among the
 * remaining ones (in order) the first with the strictly largest count_common (position 0 when all
 * counts are zero), remove it, pair the two.  pairs_first[p] / pairs_second[p] receive the dataset
 * ids of pair p in processing order; second = UINT64_MAX for the unpaired last leaf.  Returns the
 * number of pairs. */
size_t orc_scaffold_pairs(OrcMinHash *const *leaves, size_t n, uint64_t *pairs_first, uint64_t *pairs_second) {
    size_t *alive = (size_t *)malloc((n ? n : 1) * sizeof(size_t));
    size_t n_alive = n, n_pairs = 0;
    for (size_t i = 0; i < n; i++) alive[i] = i;
    while (n_alive) {
        const size_t next = alive[--n_alive];
        if (n_alive == 0) {
            pairs_first[n_pairs] = next;
            pairs_second[n_pairs++] = UINT64_MAX;
            break;
        }
        size_t similar_pos = 0;
        uint64_t current_max = 0;
        for (size_t pos = 0; pos < n_alive; pos++) {
            uint64_t common = 0;
            orc_mh_count_common(leaves[next], leaves[alive[pos]], &common);
            if (common > current_max) { current_max = common; similar_pos = pos; }
        }
        pairs_first[n_pairs] = next;
        pairs_second[n_pairs++] = alive[similar_pos];
        memmove(alive + similar_pos, alive + similar_pos + 1, (n_alive - similar_pos - 1) * sizeof(size_t));
        n_alive--;
    }
    free(alive);
    return n_pairs;
}
/* reads of fixed length laid out back to back; every read is one add_sequence */
int orc_mh_add_reads(OrcMinHash *mh, const uint8_t *buf, size_t nreads, size_t readlen, int force) {
    for (size_t r = 0; r < nreads; r++) {
        int e = orc_mh_add_sequence(mh, buf + r * readlen, readlen, force, NULL);
        if (e) return e;
    }
    return ORC_OK;
}

/* ------------------------------------------------------------------ */
/* MD5 (RFC 1321) -- needed for md5sum (lib.rs:72-77,86)                */
/* ------------------------------------------------------------------ */
typedef struct {
    uint32_t a, b, c, d;
    uint64_t nbytes;
    uint8_t buf[64];
    size_t fill;
} md5ctx;
static const uint32_t MD5_K[64] = {
    0xd76aa478, 0xe8c7b756, 0x242070db, 0xc1bdceee, 0xf57c0faf, 0x4787c62a, 0xa8304613, 0xfd469501,
    0x698098d8, 0x8b44f7af, 0xffff5bb1, 0x895cd7be, 0x6b901122, 0xfd987193, 0xa679438e, 0x49b40821,
    0xf61e2562, 0xc040b340, 0x265e5a51, 0xe9b6c7aa, 0xd62f105d, 0x02441453, 0xd8a1e681, 0xe7d3fbc8,
    0x21e1cde6, 0xc33707d6, 0xf4d50d87, 0x455a14ed, 0xa9e3e905, 0xfcefa3f8, 0x676f02d9, 0x8d2a4c8a,
    0xfffa3942, 0x8771f681, 0x6d9d6122, 0xfde5380c, 0xa4beea44, 0x4bdecfa9, 0xf6bb4b60, 0xbebfbc70,
    0x289b7ec6, 0xeaa127fa, 0xd4ef3085, 0x04881d05, 0xd9d4d039, 0xe6db99e5, 0x1fa27cf8, 0xc4ac5665,
    0xf4292244, 0x432aff97, 0xab9423a7, 0xfc93a039, 0x655b59c3, 0x8f0ccc92, 0xffeff47d, 0x85845dd1,
    0x6fa87e4f, 0xfe2ce6e0, 0xa3014314, 0x4e0811a1, 0xf7537e82, 0xbd3af235, 0x2ad7d2bb, 0xeb86d391};
static const uint8_t MD5_S[64] = {7, 12, 17, 22, 7, 12, 17, 22, 7, 12, 17, 22, 7, 12, 17, 22,
                                  5, 9,  14, 20, 5, 9,  14, 20, 5, 9,  14, 20, 5, 9,  14, 20,
                                  4, 11, 16, 23, 4, 11, 16, 23, 4, 11, 16, 23, 4, 11, 16, 23,
                                  6, 10, 15, 21, 6, 10, 15, 21, 6, 10, 15, 21, 6, 10, 15, 21};
static void md5_block(md5ctx *c, const uint8_t *p) {
    uint32_t m[16], a = c->a, b = c->b, cc = c->c, d = c->d;
    for (int i = 0; i < 16; i++)
        m[i] = (uint32_t)p[4 * i] | ((uint32_t)p[4 * i + 1] << 8) | ((uint32_t)p[4 * i + 2] << 16) |
               ((uint32_t)p[4 * i + 3] << 24);
    for (int i = 0; i < 64; i++) {
        uint32_t f; int g;
        if (i < 16) { f = (b & cc) | (~b & d); g = i; }
        else if (i < 32) { f = (d & b) | (~d & cc); g = (5 * i + 1) & 15; }
        else if (i < 48) { f = b ^ cc ^ d; g = (3 * i + 5) & 15; }
        else { f = cc ^ (b | ~d); g = (7 * i) & 15; }
        uint32_t t = a + f + MD5_K[i] + m[g];
        a = d; d = cc; cc = b;
        b = b + ((t << MD5_S[i]) | (t >> (32 - MD5_S[i])));
    }
    c->a += a; c->b += b; c->c += cc; c->d += d;
}
static void md5_init(md5ctx *c) {
    c->a = 0x67452301; c->b = 0xefcdab89; c->c = 0x98badcfe; c->d = 0x10325476;
    c->nbytes = 0; c->fill = 0;
}
static void md5_update(md5ctx *c, const void *data, size_t n) {
    const uint8_t *p = (const uint8_t *)data;
    c->nbytes += n;
    while (n) {
        size_t t = 64 - c->fill; if (t > n) t = n;
        memcpy(c->buf + c->fill, p, t);
        c->fill += t; p += t; n -= t;
        if (c->fill == 64) { md5_block(c, c->buf); c->fill = 0; }
    }
}
static void md5_final(md5ctx *c, uint8_t out[16]) {
    uint64_t bits = c->nbytes * 8;
    uint8_t pad = 0x80;
    md5_update(c, &pad, 1);
    pad = 0;
    while (c->fill != 56) md5_update(c, &pad, 1);
    uint8_t lenb[8];
    for (int i = 0; i < 8; i++) lenb[i] = (uint8_t)(bits >> (8 * i));
    md5_update(c, lenb, 8);
    uint32_t w[4] = {c->a, c->b, c->c, c->d};
    for (int i = 0; i < 4; i++)
        for (int j = 0; j < 4; j++) out[4 * i + j] = (uint8_t)(w[i] >> (8 * j));
}
/* generic md5 of a buffer -> 32 hex chars + NUL (pinned by RFC 1321 vectors in the tests) */
void orc_md5_hex(const uint8_t *data, size_t n, char out[33]) {
    md5ctx c; uint8_t d[16];
    md5_init(&c); md5_update(&c, data, n); md5_final(&c, d);
    for (int i = 0; i < 16; i++) snprintf(out + 2 * i, 3, "%02x", d[i]);
}

/* lib.rs:72-77,86: md5 over ksize.to_string() then every min.to_string(), no separators */
void orc_mh_md5sum(const OrcMinHash *mh, char out[33]) {
    md5ctx c; uint8_t d[16]; char t[24];
    md5_init(&c);
    int n = snprintf(t, sizeof t, "%u", mh->ksize);
    md5_update(&c, t, (size_t)n);
    for (size_t i = 0; i < mh->mins.len; i++) {
        n = snprintf(t, sizeof t, "%llu", (unsigned long long)mh->mins.p[i]);
        md5_update(&c, t, (size_t)n);
    }
    md5_final(&c, d);
    for (int i = 0; i < 16; i++) snprintf(out + 2 * i, 3, "%02x", d[i]);
}

/* ------------------------------------------------------------------ */
/* JSON output (lib.rs:62-102 KmerMinHash; :546-565 Signature; compact  */
/* serde_json::to_string, ffi.rs:498,531)                               */
/* ------------------------------------------------------------------ */
static void json_str(sbuf *s, const char *v) { /* serde_json string escaping */
    s_puts(s, "\"");
    for (const unsigned char *p = (const unsigned char *)v; *p; p++) {
        char t[8];
        switch (*p) {
        case '"': s_puts(s, "\\\""); break;
        case '\\': s_puts(s, "\\\\"); break;
        case '\b': s_puts(s, "\\b"); break;
        case '\f': s_puts(s, "\\f"); break;
        case '\n': s_puts(s, "\\n"); break;
        case '\r': s_puts(s, "\\r"); break;
        case '\t': s_puts(s, "\\t"); break;
        default:
            if (*p < 0x20) { snprintf(t, sizeof t, "\\u%04x", *p); s_puts(s, t); }
            else s_put(s, (const char *)p, 1);
        }
    }
    s_puts(s, "\"");
}
static void json_u64_array(sbuf *s, const vec64 *v) {
    s_puts(s, "[");
    for (size_t i = 0; i < v->len; i++) { if (i) s_puts(s, ","); s_putu(s, v->p[i]); }
    s_puts(s, "]");
}
/* shortest round-trip decimal for an f64, ryu-style layout for the common range */
static void json_f64(sbuf *s, double x) {
    char t[40];
    if (!isfinite(x)) { s_puts(s, "null"); return; }
    for (int prec = 1; prec <= 17; prec++) {
        snprintf(t, sizeof t, "%.*g", prec, x);
        if (strtod(t, NULL) == x) break;
    }
    if (!strpbrk(t, ".eEn")) strcat(t, ".0");
    s_puts(s, t);
}
static void json_minhash(sbuf *s, const OrcMinHash *mh) {
    char md5[33];
    orc_mh_md5sum(mh, md5);
    s_puts(s, "{\"num\":"); s_putu(s, mh->num);
    s_puts(s, ",\"ksize\":"); s_putu(s, mh->ksize);
    s_puts(s, ",\"seed\":"); s_putu(s, mh->seed);
    s_puts(s, ",\"max_hash\":"); s_putu(s, mh->max_hash);
    s_puts(s, ",\"mins\":"); json_u64_array(s, &mh->mins);
    s_puts(s, ",\"md5sum\":\""); s_puts(s, md5); s_puts(s, "\"");
    if (mh->has_abunds) { s_puts(s, ",\"abundances\":"); json_u64_array(s, &mh->abunds); }
    s_puts(s, ",\"molecule\":"); s_puts(s, mh->is_protein ? "\"protein\"" : "\"DNA\"");
    s_puts(s, "}");
}

/* Signature::default() (lib.rs:648-661) + name/filename (NULL => null) around n sketches.
 * Returns a malloc'ed NUL-terminated string; free with orc_free. */
char *orc_signature_json(const char *name, const char *filename, OrcMinHash *const *mhs, size_t n) {
    sbuf s = {0};
    s_puts(&s, "{\"class\":\"sourmash_signature\",\"email\":\"\",\"hash_function\":\"0.murmur64\",\"filename\":");
    if (filename) json_str(&s, filename); else s_puts(&s, "null");
    s_puts(&s, ",\"name\":");
    if (name) json_str(&s, name); else s_puts(&s, "null");
    s_puts(&s, ",\"license\":\"CC0\",\"signatures\":[");
    for (size_t i = 0; i < n; i++) { if (i) s_puts(&s, ","); json_minhash(&s, mhs[i]); }
    s_puts(&s, "],\"version\":");
    json_f64(&s, 0.4);
    s_puts(&s, "}");
    return s.p;
}
void orc_free(void *p) { free(p); }

/* ===========================================================================================
 * Nodegraph (khmer bloom filter) -- src/index/nodegraph.rs:11-225 -- and SBT::find
 * (src/index/sbt.rs:147-175) with the Node<Nodegraph> x Leaf<Signature> comparisons
 * (src/index/sbt.rs:233-277).  SURVEY 8(f) rank 3.  FixedBitSet = u32 blocks, bit i at block i / 32,
 * bit i % 32.
 * =========================================================================================== */
typedef struct OrcNodegraph {
    size_t n_tables;
    size_t *len;       /* bits per table */
    uint32_t **bs;     /* ceil(len / 32) blocks per table */
    size_t ksize, occupied_bins, unique_kmers;
} OrcNodegraph;

/* Nodegraph::new, nodegraph.rs:20-32 */
OrcNodegraph *orc_ng_new(const uint64_t *tablesizes, size_t n_tables, size_t ksize) {
    OrcNodegraph *ng = (OrcNodegraph *)calloc(1, sizeof *ng);
    ng->n_tables = n_tables;
    ng->len = (size_t *)calloc(n_tables ? n_tables : 1, sizeof(size_t));
    ng->bs = (uint32_t **)calloc(n_tables ? n_tables : 1, sizeof(uint32_t *));
    for (size_t t = 0; t < n_tables; t++) {
        ng->len[t] = (size_t)tablesizes[t];
        ng->bs[t] = (uint32_t *)calloc((ng->len[t] + 31) / 32 + 1, sizeof(uint32_t));
    }
    ng->ksize = ksize;
    return ng;
}
void orc_ng_free(OrcNodegraph *ng) {
    if (!ng) return;
    for (size_t t = 0; t < ng->n_tables; t++) free(ng->bs[t]);
    free(ng->bs); free(ng->len); free(ng);
}
static int ng_put(uint32_t *bs, size_t bit) { /* FixedBitSet::put: sets, returns the previous value */
    const uint32_t m = 1u << (bit & 31);
    const int prev = (bs[bit >> 5] & m) != 0;
    bs[bit >> 5] |= m;
    return prev;
}
/* Nodegraph::count, nodegraph.rs:34-50 */
int orc_ng_count(OrcNodegraph *ng, uint64_t hash) {
    int is_new = 0;
    for (size_t t = 0; t < ng->n_tables; t++) {
        const uint64_t bin = hash % (uint64_t)ng->len[t];
        if (!ng_put(ng->bs[t], (size_t)bin)) { ng->occupied_bins += 1; is_new = 1; }
    }
    if (is_new) ng->unique_kmers += 1;
    return is_new;
}
/* Nodegraph::get, nodegraph.rs:52-60 */
size_t orc_ng_get(const OrcNodegraph *ng, uint64_t hash) {
    for (size_t t = 0; t < ng->n_tables; t++) {
        const uint64_t bin = hash % (uint64_t)ng->len[t];
        if (!(ng->bs[t][bin >> 5] & (1u << (bin & 31)))) return 0;
    }
    return 1;
}
/* count / get over a batch in one call: is_new[i] = count(hashes[i]) in batch order, present[i] = get(hashes[i]);
 * either output may be NULL.  Return the sums. */
uint64_t orc_ng_count_many(OrcNodegraph *ng, const uint64_t *hashes, size_t n, uint8_t *is_new) {
    uint64_t sum = 0;
    for (size_t i = 0; i < n; i++) {
        const int v = orc_ng_count(ng, hashes[i]);
        if (is_new) is_new[i] = (uint8_t)v;
        sum += (uint64_t)v;
    }
    return sum;
}
uint64_t orc_ng_get_many(const OrcNodegraph *ng, const uint64_t *hashes, size_t n, uint8_t *present) {
    uint64_t sum = 0;
    for (size_t i = 0; i < n; i++) {
        const size_t v = orc_ng_get(ng, hashes[i]);
        if (present) present[i] = (uint8_t)v;
        sum += v;
    }
    return sum;
}
/* Nodegraph::update, nodegraph.rs:63-91 (occupied_bins deliberately not updated there).
 * Returns -1 where the reference would panic (a set bit of `other` beyond self's table). */
int orc_ng_update(OrcNodegraph *ng, const OrcNodegraph *other) {
    const size_t nt = ng->n_tables < other->n_tables ? ng->n_tables : other->n_tables; /* zip */
    for (size_t t = 0; t < nt; t++)
        for (size_t x = 0; x < other->len[t]; x++)
            if (other->bs[t][x >> 5] & (1u << (x & 31))) {
                if (x >= ng->len[t]) return -1;
                ng_put(ng->bs[t], x);
            }
    return 0;
}
/* Nodegraph::save_to_writer, nodegraph.rs:99-133; returns the byte count, writes when it fits */
size_t orc_ng_save(const OrcNodegraph *ng, uint8_t *out, size_t cap) {
    size_t n = 0;
#define NG_PUT8(v) do { if (n < cap) out[n] = (uint8_t)(v); n++; } while (0)
#define NG_PUTLE(v, bytes) do { uint64_t _v = (uint64_t)(v); for (int _b = 0; _b < (bytes); _b++) NG_PUT8(_v >> (8 * _b)); } while (0)
    NG_PUT8('O'); NG_PUT8('X'); NG_PUT8('L'); NG_PUT8('I');
    NG_PUT8(4);                         /* version */
    NG_PUT8(2);                         /* ht_type */
    NG_PUTLE(ng->ksize, 4);
    NG_PUT8(ng->n_tables);
    NG_PUTLE(ng->occupied_bins, 8);
    for (size_t t = 0; t < ng->n_tables; t++) {
        const size_t len = ng->len[t], blocks = (len + 31) / 32;
        NG_PUTLE(len, 8);
        for (size_t i = 0; i < blocks; i++) {
            const uint32_t chunk = ng->bs[t][i];
            const size_t next = (i + 1) * 32;
            if (next <= len) {
                NG_PUTLE(chunk, 4);
            } else {
                const size_t rem = len - i * 32;
                const size_t remainder = (rem % 8 != 0) ? rem / 8 + 1 : rem / 8;
                if (remainder == 0) NG_PUT8(0);
                else for (size_t pos = 0; pos < remainder; pos++) NG_PUT8((chunk >> (pos * 8)) & 0xff);
            }
        }
    }
#undef NG_PUT8
#undef NG_PUTLE
    return n;
}
/* Nodegraph::from_reader, nodegraph.rs:135-181; NULL where the reference's asserts / reads fail */
OrcNodegraph *orc_ng_load(const uint8_t *d, size_t n) {
    size_t p = 0;
    if (n < 19) return NULL;
    if (!(d[0] == 0x4f && d[1] == 0x58 && d[2] == 0x4c && d[3] == 0x49)) return NULL;
    if (d[4] != 0x04 || d[5] != 0x02) return NULL;
    const uint32_t ksize = (uint32_t)d[6] | ((uint32_t)d[7] << 8) | ((uint32_t)d[8] << 16) | ((uint32_t)d[9] << 24);
    const size_t n_tables = d[10];
    uint64_t occ = 0;
    for (int b = 0; b < 8; b++) occ |= (uint64_t)d[11 + b] << (8 * b);
    p = 19;
    uint64_t *sizes = (uint64_t *)calloc(n_tables ? n_tables : 1, sizeof(uint64_t));
    /* first pass over the table headers to size the bitsets */
    size_t q = p;
    for (size_t t = 0; t < n_tables; t++) {
        if (q + 8 > n) { free(sizes); return NULL; }
        uint64_t ts = 0;
        for (int b = 0; b < 8; b++) ts |= (uint64_t)d[q + b] << (8 * b);
        sizes[t] = ts;
        q += 8 + (size_t)(ts / 8 + 1);
        if (q > n) { free(sizes); return NULL; }
    }
    OrcNodegraph *ng = orc_ng_new(sizes, n_tables, ksize);
    free(sizes);
    for (size_t t = 0; t < n_tables; t++) {
        const size_t tablesize = ng->len[t], byte_size = tablesize / 8 + 1;
        p += 8;
        for (size_t pos = 0; pos < byte_size; pos++) {
            const uint8_t byte = d[p++];
            if (byte == 0) continue;
            for (unsigned i = 0; i < 8; i++)
                if (byte & (1u << i)) {
                    const size_t bit = pos * 8 + i;
                    if (bit >= tablesize) { orc_ng_free(ng); return NULL; } /* FixedBitSet::insert panics */
                    ng->bs[t][bit >> 5] |= 1u << (bit & 31);
                }
        }
    }
    ng->occupied_bins = (size_t)occ;
    ng->unique_kmers = 0; /* "a khmer issue, it doesn't save unique_kmers" */
    return ng;
}
size_t orc_ng_n_tables(const OrcNodegraph *ng) { return ng->n_tables; }
uint64_t orc_ng_tablesize(const OrcNodegraph *ng, size_t t) { return ng->len[t]; }
size_t orc_ng_ksize(const OrcNodegraph *ng) { return ng->ksize; }
size_t orc_ng_occupied_bins(const OrcNodegraph *ng) { return ng->occupied_bins; }
size_t orc_ng_unique_kmers(const OrcNodegraph *ng) { return ng->unique_kmers; }
const uint32_t *orc_ng_blocks(const OrcNodegraph *ng, size_t t) { return ng->bs[t]; }
static void ng_and_or_counts(const OrcNodegraph *a, const OrcNodegraph *b, size_t *n_and, size_t *n_or) {
    /* FixedBitSet::intersection / union walk the set bits of the operands; over tables of equal
     * length that is a popcount of AND / OR (bits beyond len are never set) */
    const size_t nt = a->n_tables < b->n_tables ? a->n_tables : b->n_tables;
    *n_and = 0; *n_or = 0;
    for (size_t t = 0; t < nt; t++) {
        const size_t ba = (a->len[t] + 31) / 32, bb = (b->len[t] + 31) / 32, lo = ba < bb ? ba : bb;
        for (size_t i = 0; i < lo; i++) {
            *n_and += (size_t)__builtin_popcount(a->bs[t][i] & b->bs[t][i]);
            *n_or += (size_t)__builtin_popcount(a->bs[t][i] | b->bs[t][i]);
        }
        for (size_t i = lo; i < ba; i++) *n_or += (size_t)__builtin_popcount(a->bs[t][i]);
        for (size_t i = lo; i < bb; i++) *n_or += (size_t)__builtin_popcount(b->bs[t][i]);
    }
}
/* Nodegraph::similarity, nodegraph.rs:199-213 */
double orc_ng_similarity(const OrcNodegraph *a, const OrcNodegraph *b) {
    size_t x, u;
    ng_and_or_counts(a, b, &x, &u);
    return (double)x / (double)u;
}
/* Nodegraph::containment, nodegraph.rs:215-224: the denominator is the total table LENGTH of self */
double orc_ng_containment(const OrcNodegraph *a, const OrcNodegraph *b) {
    size_t x, u, size = 0;
    ng_and_or_counts(a, b, &x, &u);
    for (size_t t = 0; t < a->n_tables; t++) size += a->len[t];
    return (double)x / (double)size;
}
/* sum of get(h) over a sketch's mins: the numerator of Node<Nodegraph> x Leaf<Signature>, sbt.rs:245,266 */
uint64_t orc_ng_matches(const OrcNodegraph *ng, const OrcMinHash *mh) {
    uint64_t m = 0;
    for (size_t i = 0; i < mh->mins.len; i++) m += orc_ng_get(ng, mh->mins.p[i]);
    return m;
}
/* Comparable<Leaf<Signature>> for Node<Nodegraph>, sbt.rs:233-277 */
double orc_node_similarity(const OrcNodegraph *ng, uint64_t min_n_below, const OrcMinHash *query) {
    if (query->mins.len == 0) return 0.0;
    return (double)orc_ng_matches(ng, query) / (double)min_n_below;
}
double orc_node_containment(const OrcNodegraph *ng, const OrcMinHash *query) {
    if (query->mins.len == 0) return 0.0;
    return (double)orc_ng_matches(ng, query) / (double)query->mins.len;
}
/* SBT::find, sbt.rs:147-175, with search_minhashes (mode 0) / search_minhashes_containment (mode 1),
 * search.rs:3-9.  Nodes and leaves are given by tree position; hits_pos receives the positions of the
 * matching leaves in the order the depth-first walk meets them (children are pushed 0..d-1 and popped
 * from the back, so the LAST child is visited first).
 * orc_sbt_new indexes a tree once for many queries (orc_sbt_query); it copies the position and pointer arrays
 * but borrows the Nodegraphs and sketches, which must outlive it.  A position listed twice resolves to its
 * first entry, as a map built by inserting the entries in order and keeping the first. */
typedef struct { uint64_t pos; size_t idx; } PosIdx;
typedef struct OrcSbt {
    uint32_t d;
    size_t n_nodes, n_leaves;
    PosIdx *node_at, *leaf_at; /* sorted by (position, index) */
    OrcNodegraph **nodes;
    uint64_t *min_n_below;
    OrcMinHash **leaves;
} OrcSbt;
static int pos_idx_cmp(const void *a, const void *b) {
    const PosIdx *x = (const PosIdx *)a, *y = (const PosIdx *)b;
    if (x->pos != y->pos) return x->pos < y->pos ? -1 : 1;
    return x->idx < y->idx ? -1 : x->idx > y->idx;
}
static PosIdx *pos_index(const uint64_t *pos, size_t n) {
    PosIdx *a = (PosIdx *)malloc((n ? n : 1) * sizeof(PosIdx));
    for (size_t i = 0; i < n; i++) { a[i].pos = pos[i]; a[i].idx = i; }
    qsort(a, n, sizeof(PosIdx), pos_idx_cmp);
    return a;
}
/* index of the first entry at `pos`, n when there is none */
static size_t pos_lookup(const PosIdx *a, size_t n, uint64_t pos) {
    size_t lo = 0, hi = n;
    while (lo < hi) {
        const size_t mid = lo + (hi - lo) / 2;
        if (a[mid].pos < pos) lo = mid + 1; else hi = mid;
    }
    return (lo < n && a[lo].pos == pos) ? a[lo].idx : n;
}
static void *copy_array(const void *p, size_t n, size_t size) {
    void *q = malloc((n ? n : 1) * size);
    if (n) memcpy(q, p, n * size);
    return q;
}
OrcSbt *orc_sbt_new(uint32_t d, const uint64_t *node_pos, OrcNodegraph *const *nodes, const uint64_t *min_n_below,
                    size_t n_nodes, const uint64_t *leaf_pos, OrcMinHash *const *leaves, size_t n_leaves) {
    OrcSbt *t = (OrcSbt *)calloc(1, sizeof *t);
    t->d = d;
    t->n_nodes = n_nodes;
    t->n_leaves = n_leaves;
    t->node_at = pos_index(node_pos, n_nodes);
    t->leaf_at = pos_index(leaf_pos, n_leaves);
    t->nodes = (OrcNodegraph **)copy_array(nodes, n_nodes, sizeof *nodes);
    t->min_n_below = (uint64_t *)copy_array(min_n_below, n_nodes, sizeof *min_n_below);
    t->leaves = (OrcMinHash **)copy_array(leaves, n_leaves, sizeof *leaves);
    return t;
}
void orc_sbt_free(OrcSbt *t) {
    if (!t) return;
    free(t->node_at); free(t->leaf_at); free(t->nodes); free(t->min_n_below); free(t->leaves); free(t);
}
size_t orc_sbt_query(const OrcSbt *t, const OrcMinHash *query, int mode, double threshold, uint64_t *hits_pos) {
    size_t n_hits = 0, cap = 64, top = 0;
    uint64_t *stack = (uint64_t *)malloc(cap * sizeof(uint64_t));
    stack[top++] = 0;
    while (top) {
        const uint64_t pos = stack[--top];
        /* positions are unique in a d-ary heap layout, so the reference's `visited` set never fires */
        const size_t ni = pos_lookup(t->node_at, t->n_nodes, pos);
        if (ni < t->n_nodes) {
            const double v = mode ? orc_node_containment(t->nodes[ni], query)
                                  : orc_node_similarity(t->nodes[ni], t->min_n_below[ni], query);
            if (v > threshold) {
                for (uint32_t c = 0; c < t->d; c++) {
                    if (top == cap) { cap *= 2; stack = (uint64_t *)realloc(stack, cap * sizeof(uint64_t)); }
                    stack[top++] = (uint64_t)t->d * pos + c + 1;
                }
            }
            continue;
        }
        const size_t li = pos_lookup(t->leaf_at, t->n_leaves, pos);
        if (li < t->n_leaves) {
            const double v = mode ? orc_leaf_containment(t->leaves[li], query) : orc_leaf_similarity(t->leaves[li], query);
            if (v > threshold) hits_pos[n_hits++] = pos;
        }
    }
    free(stack);
    return n_hits;
}
