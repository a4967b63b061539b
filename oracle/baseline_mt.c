/*
 * baseline_mt.c -- the CPU baseline legs of bench.py (cpu_baseline and
 * --impl reference): the oracle's reference-faithful algorithm run over
 * independent units (reads / matrix rows) on all host threads.
 *
 * TEST / MEASUREMENT INFRASTRUCTURE ONLY (see oracle.c header).  The reference
 * itself is single-threaded (no rayon/threads anywhere in /root/reference/src);
 * spreading independent add_sequence calls / compare rows over std threads is
 * the most favourable reading of "the CPU path on the box's host cores".
 */
#include <pthread.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

typedef struct OrcMinHash OrcMinHash;
OrcMinHash *orc_mh_new(uint32_t, uint32_t, int, uint64_t, uint64_t, int);
void orc_mh_free(OrcMinHash *);
int orc_mh_add_sequence(OrcMinHash *, const uint8_t *, size_t, int, char *);
int orc_mh_merge(OrcMinHash *, const OrcMinHash *);
int orc_mh_intersection_size(const OrcMinHash *, const OrcMinHash *, uint64_t *, uint64_t *);
size_t orc_mh_size(const OrcMinHash *);

typedef struct {
    const uint8_t *buf;
    size_t r0, r1, readlen;
    const uint32_t *ksizes;
    int nk;
    uint32_t num;
    uint64_t max_hash;
    int track;
    OrcMinHash **out; /* nk sketches */
} sketch_job;

static void *sketch_worker(void *arg) {
    sketch_job *j = (sketch_job *)arg;
    for (int q = 0; q < j->nk; q++)
        j->out[q] = orc_mh_new(j->num, j->ksizes[q], 0, 42, j->max_hash, j->track);
    for (size_t r = j->r0; r < j->r1; r++)
        for (int q = 0; q < j->nk; q++)
            orc_mh_add_sequence(j->out[q], j->buf + r * j->readlen, j->readlen, 1, NULL);
    return NULL;
}

/* Sketch nreads fixed-length reads into nk sketches (one per ksize), reads
 * block-partitioned over nthreads, per-thread sketches combined with merge
 * (lib.rs:307-403).  Returns the combined sketches in out[nk] (caller frees). */
void orc_mt_sketch_reads(const uint8_t *buf, size_t nreads, size_t readlen, const uint32_t *ksizes, int nk,
                         uint32_t num, uint64_t max_hash, int track, int nthreads, OrcMinHash **out) {
    if (nthreads < 1) nthreads = 1;
    pthread_t *th = (pthread_t *)malloc(sizeof(pthread_t) * (size_t)nthreads);
    sketch_job *jobs = (sketch_job *)calloc((size_t)nthreads, sizeof(sketch_job));
    for (int t = 0; t < nthreads; t++) {
        jobs[t].buf = buf; jobs[t].readlen = readlen;
        jobs[t].r0 = nreads * (size_t)t / (size_t)nthreads;
        jobs[t].r1 = nreads * (size_t)(t + 1) / (size_t)nthreads;
        jobs[t].ksizes = ksizes; jobs[t].nk = nk; jobs[t].num = num;
        jobs[t].max_hash = max_hash; jobs[t].track = track;
        jobs[t].out = (OrcMinHash **)calloc((size_t)nk, sizeof(OrcMinHash *));
        pthread_create(&th[t], NULL, sketch_worker, &jobs[t]);
    }
    for (int t = 0; t < nthreads; t++) pthread_join(th[t], NULL);
    for (int q = 0; q < nk; q++) {
        out[q] = jobs[0].out[q];
        for (int t = 1; t < nthreads; t++) {
            orc_mh_merge(out[q], jobs[t].out[q]);
            orc_mh_free(jobs[t].out[q]);
        }
    }
    for (int t = 0; t < nthreads; t++) free(jobs[t].out);
    free(jobs); free(th);
}

typedef struct {
    const uint8_t *buf;
    const uint64_t *offsets;
    size_t n_seqs;
    uint32_t num, ksize;
    int is_protein, track;
    uint64_t seed, max_hash;
    size_t *next; /* shared: the next sequence to take */
    OrcMinHash **out;
} each_job;

static void *each_worker(void *arg) {
    each_job *j = (each_job *)arg;
    for (;;) {
        const size_t s = __atomic_fetch_add(j->next, 1, __ATOMIC_RELAXED);
        if (s >= j->n_seqs) return NULL;
        OrcMinHash *mh = orc_mh_new(j->num, j->ksize, j->is_protein, j->seed, j->max_hash, j->track);
        orc_mh_add_sequence(mh, j->buf + j->offsets[s], (size_t)(j->offsets[s + 1] - j->offsets[s]), 1, NULL);
        j->out[s] = mh;
    }
}

/* One fresh sketch per sequence buf[offsets[s]:offsets[s+1]] (KmerMinHash::new + add_sequence(force = true)), the
 * sequences taken one at a time by nthreads host threads: the reference loop behind a sketch collection
 * (lib.rs:142-174, 252-305).  out[s] receives sequence s's sketch (caller frees). */
void orc_mt_sketch_each(const uint8_t *buf, const uint64_t *offsets, size_t n_seqs, uint32_t num, uint32_t ksize,
                        int is_protein, uint64_t seed, uint64_t max_hash, int track, int nthreads, OrcMinHash **out) {
    if (nthreads < 1) nthreads = 1;
    size_t next = 0;
    pthread_t *th = (pthread_t *)malloc(sizeof(pthread_t) * (size_t)nthreads);
    each_job job = {buf, offsets, n_seqs, num, ksize, is_protein, track, seed, max_hash, &next, out};
    for (int t = 0; t < nthreads; t++) pthread_create(&th[t], NULL, each_worker, &job);
    for (int t = 0; t < nthreads; t++) pthread_join(th[t], NULL);
    free(th);
}

typedef struct {
    OrcMinHash *const *rows; OrcMinHash *const *cols;
    size_t i0, i1, nc;
    uint32_t *common, *size;
} cmp_job;

static void *cmp_worker(void *arg) {
    cmp_job *j = (cmp_job *)arg;
    for (size_t i = j->i0; i < j->i1; i++)
        for (size_t c = 0; c < j->nc; c++) {
            uint64_t cm, sz;
            orc_mh_intersection_size(j->rows[i], j->cols[c], &cm, &sz);
            j->common[i * j->nc + c] = (uint32_t)cm;
            j->size[i * j->nc + c] = (uint32_t)sz;
        }
    return NULL;
}

/* all rows x all cols KmerMinHash::compare integer parts, rows split over threads */
void orc_mt_compare_matrix(OrcMinHash *const *rows, size_t nr, OrcMinHash *const *cols, size_t nc,
                           uint32_t *common, uint32_t *size, int nthreads) {
    if (nthreads < 1) nthreads = 1;
    pthread_t *th = (pthread_t *)malloc(sizeof(pthread_t) * (size_t)nthreads);
    cmp_job *jobs = (cmp_job *)calloc((size_t)nthreads, sizeof(cmp_job));
    for (int t = 0; t < nthreads; t++) {
        jobs[t].rows = rows; jobs[t].cols = cols; jobs[t].nc = nc;
        jobs[t].i0 = nr * (size_t)t / (size_t)nthreads;
        jobs[t].i1 = nr * (size_t)(t + 1) / (size_t)nthreads;
        jobs[t].common = common; jobs[t].size = size;
        pthread_create(&th[t], NULL, cmp_worker, &jobs[t]);
    }
    for (int t = 0; t < nthreads; t++) pthread_join(th[t], NULL);
    free(jobs); free(th);
}

typedef struct {
    OrcMinHash *const *mhs;
    const uint64_t *ia, *ib;
    size_t p0, p1;
    uint32_t *common, *size;
} pair_job;

static void *pair_worker(void *arg) {
    pair_job *j = (pair_job *)arg;
    for (size_t p = j->p0; p < j->p1; p++) {
        uint64_t cm, sz;
        orc_mh_intersection_size(j->mhs[j->ia[p]], j->mhs[j->ib[p]], &cm, &sz);
        j->common[p] = (uint32_t)cm;
        j->size[p] = (uint32_t)sz;
    }
    return NULL;
}

/* KmerMinHash::compare integer parts of a LIST of pairs (mhs[ia[p]], mhs[ib[p]]): the sampled-pairs parity check
 * of the full-size matrix (SURVEY 8(d) cfg3), pairs split over threads */
void orc_mt_compare_pairs(OrcMinHash *const *mhs, const uint64_t *ia, const uint64_t *ib, size_t n_pairs,
                          uint32_t *common, uint32_t *size, int nthreads) {
    if (nthreads < 1) nthreads = 1;
    pthread_t *th = (pthread_t *)malloc(sizeof(pthread_t) * (size_t)nthreads);
    pair_job *jobs = (pair_job *)calloc((size_t)nthreads, sizeof(pair_job));
    for (int t = 0; t < nthreads; t++) {
        jobs[t].mhs = mhs; jobs[t].ia = ia; jobs[t].ib = ib;
        jobs[t].p0 = n_pairs * (size_t)t / (size_t)nthreads;
        jobs[t].p1 = n_pairs * (size_t)(t + 1) / (size_t)nthreads;
        jobs[t].common = common; jobs[t].size = size;
        pthread_create(&th[t], NULL, pair_worker, &jobs[t]);
    }
    for (int t = 0; t < nthreads; t++) pthread_join(th[t], NULL);
    free(jobs); free(th);
}
