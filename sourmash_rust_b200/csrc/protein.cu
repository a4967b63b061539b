// protein.cu -- the protein arm of KmerMinHash::add_sequence (reference src/lib.rs:275-302):
// every sequence is translated in its three forward frames and the three frames of its reverse
// complement (to_aa, lib.rs:776-793: codons that are not three ACGT letters are DROPPED, so the
// residue stream is compacted), and every window of ksize/3 residues is hashed with MurmurHash3
// (add_word, lib.rs:247-250).  No validity check; `force` is not consulted.
//
// Slot layout: sequence s (bytes [b, b+len)) owns the slot region [2b + 6s, 2(b+len) + 6(s+1)); inside
// it frame f (order fw0, rc0, fw1, rc1, fw2, rc2 -- the order the reference adds them) owns
// cap = len/3 + 1 slots, one per codon.  translate -> exclusive scan of the kept flags -> compaction
// -> one thread per kept residue hashes the window that starts there if it fits in its frame.
// The first three steps do not depend on the window size or the seed (beyond skipping sequences shorter
// than pb.ksize), so several protein sketches of one batch can share them and run only the hash step
// each; the hash step skips sequences shorter than its own pb.ksize.
#include "device.hpp"
#include "kernels.cuh"
#include "murmur3.cuh"

namespace smb200 {

__device__ __forceinline__ void pr_seq(const ProteinBatch &pb, uint64_t s, uint64_t &begin, uint64_t &len) {
    if (pb.offsets) { begin = pb.offsets[s]; len = pb.offsets[s + 1] - begin; }
    else if (pb.read_len) { begin = s * (uint64_t)pb.read_len; len = pb.read_len; }
    else { begin = 0; len = pb.n; }
}
// sequence owning slot t
__device__ __forceinline__ uint64_t pr_find(const ProteinBatch &pb, uint64_t t) {
    if (!pb.offsets) return pb.read_len ? t / (2ull * pb.read_len + 6) : 0;
    uint64_t lo = 0, hi = pb.n_seqs;  // last s with region(s) <= t
    while (hi - lo > 1) {
        const uint64_t mid = (lo + hi) >> 1;
        if (2 * pb.offsets[mid] + 6 * mid <= t) lo = mid; else hi = mid;
    }
    return lo;
}
__device__ __forceinline__ int pr_code(uint8_t c) {  // upper-cased ACGT -> 0..3, anything else -> -1
    c = (c >= 'a' && c <= 'z') ? (uint8_t)(c - 32) : c;  // lib.rs:253-256
    return c == 'A' ? 0 : c == 'C' ? 1 : c == 'G' ? 2 : c == 'T' ? 3 : -1;
}

// CODONTABLE (lib.rs:691-763), index 16a + 4b + c with A0 C1 G2 T3
__constant__ char c_codon[65] = "KNKNTTTTRSRSIIMIQHQHPPPPRRRRLLLLEDEDAAAAGGGGVVVV*Y*YSSSS*CWCLFLF";

__global__ void __launch_bounds__(256) protein_translate_kernel(const ProteinBatch pb, uint64_t total, uint8_t *aa,
                                                                uint64_t *flags) {
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; t <= total; t += stride) {
        uint8_t out = 0;
        if (t < total) {
            const uint64_t s = pr_find(pb, t);
            uint64_t begin, len;
            pr_seq(pb, s, begin, len);
            const uint64_t local = t - (2 * begin + 6 * s), cap = len / 3 + 1;
            const uint64_t f = local / cap, j = local - f * cap;
            if (f < 6 && len >= pb.ksize) {
                const uint64_t i = f >> 1, start = i + 3 * j;
                if (start + 3 <= len) {
                    int c[3];
                    if (!(f & 1)) {
#pragma unroll
                        for (int q = 0; q < 3; q++) c[q] = pr_code(pb.buf[begin + start + q]);
                    } else {  // revcomp (lib.rs:677-689): reversed, A<->T, C<->G
#pragma unroll
                        for (int q = 0; q < 3; q++) {
                            const int v = pr_code(pb.buf[begin + len - 1 - (start + q)]);
                            c[q] = v < 0 ? -1 : 3 - v;
                        }
                    }
                    if (c[0] >= 0 && c[1] >= 0 && c[2] >= 0) out = (uint8_t)c_codon[16 * c[0] + 4 * c[1] + c[2]];
                }
            }
        }
        aa[t] = out;
        flags[t] = out != 0;
    }
}

__global__ void __launch_bounds__(256) protein_compact_kernel(const uint8_t *__restrict__ aa,
                                                              const uint64_t *__restrict__ flags,
                                                              const uint64_t *__restrict__ pre, uint64_t total,
                                                              uint8_t *__restrict__ comp) {
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += stride)
        if (flags[t]) comp[pre[t]] = aa[t];
}

__global__ void __launch_bounds__(256) protein_hash_kernel(const ProteinBatch pb, uint64_t total,
                                                           const uint64_t *__restrict__ flags,
                                                           const uint64_t *__restrict__ pre,
                                                           const uint8_t *__restrict__ comp, const SketchOut out) {
    const uint64_t thr = *out.thr;
    const uint32_t aa_k = pb.ksize / 3;
    const int lane = threadIdx.x & 31;
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    const uint64_t rounds = (total + 31) / 32 * 32;
    for (uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; t < rounds; t += stride) {
        bool pass = false;
        uint64_t h = 0, p = 0;
        if (t < total && flags[t]) {
            const uint64_t s = pr_find(pb, t);
            uint64_t begin, len;
            pr_seq(pb, s, begin, len);
            const uint64_t region = 2 * begin + 6 * s, cap = len / 3 + 1;
            const uint64_t f = (t - region) / cap;
            const uint64_t frame_end = pre[region + (f + 1) * cap];  // kept residues before the next frame
            p = pre[t];
            if (len >= pb.ksize && p + aa_k <= frame_end) {  // a sequence shorter than ksize adds nothing
                h = murmur3_h1_bytes(comp + p, aa_k, pb.seed);
                pass = h <= thr;
            }
        }
        const unsigned bal = __ballot_sync(0xFFFFFFFFu, pass);
        if (bal) {
            unsigned long long base = 0;
            if (lane == 0) base = atomicAdd(out.counter, (unsigned long long)__popc(bal));
            base = __shfl_sync(0xFFFFFFFFu, base, 0);
            if (pass) {
                const unsigned long long idx = base + __popc(bal & ((1u << lane) - 1u));
                if (idx < out.cap) {
                    out.hash[idx] = h;
                    if (out.pos) out.pos[idx] = p;  // compacted index: the order the reference adds the words in
                }
            }
        }
    }
}

uint64_t protein_slots(uint64_t n_bytes, uint64_t n_seqs) { return 2 * n_bytes + 6 * n_seqs; }

static unsigned protein_blocks(uint64_t total) {
    const uint64_t b = (total + 255) / 256;
    return (unsigned)(b > 148 * 32 ? 148 * 32 : b);
}

void launch_protein_translate(const ProteinBatch &pb, uint8_t *aa, uint8_t *comp, uint64_t *flags, uint64_t *pre,
                              void *scan_tmp, cudaStream_t st) {
    const uint64_t total = protein_slots(pb.n, pb.n_seqs);
    if (!total) return;
    const unsigned blocks = protein_blocks(total);
    protein_translate_kernel<<<blocks, 256, 0, st>>>(pb, total, aa, flags);
    SM_LAUNCHED();
    scan_exclusive_u64(flags, pre, total + 1, scan_tmp, st);
    protein_compact_kernel<<<blocks, 256, 0, st>>>(aa, flags, pre, total, comp);
    SM_LAUNCHED();
}

void launch_protein_hash(const ProteinBatch &pb, const SketchOut &out, const uint8_t *comp, const uint64_t *flags,
                         const uint64_t *pre, cudaStream_t st) {
    const uint64_t total = protein_slots(pb.n, pb.n_seqs);
    if (!total) return;
    protein_hash_kernel<<<protein_blocks(total), 256, 0, st>>>(pb, total, flags, pre, comp, out);
    SM_LAUNCHED();
}

void launch_protein_sketch(const ProteinBatch &pb, const SketchOut &out, uint8_t *aa, uint8_t *comp, uint64_t *flags,
                           uint64_t *pre, void *scan_tmp, cudaStream_t st) {
    launch_protein_translate(pb, aa, comp, flags, pre, scan_tmp, st);
    launch_protein_hash(pb, out, comp, flags, pre, st);
}

__global__ void __launch_bounds__(256) protein_seq_starts_kernel(const uint64_t *__restrict__ offsets, uint64_t n_seqs,
                                                                 const uint64_t *__restrict__ pre, uint64_t *starts) {
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t s = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; s <= n_seqs; s += stride)
        starts[s] = pre[2 * offsets[s] + 6 * s];
}

void launch_protein_seq_starts(const uint64_t *offsets, uint64_t n_seqs, const uint64_t *pre, uint64_t *starts,
                               cudaStream_t st) {
    protein_seq_starts_kernel<<<protein_blocks(n_seqs + 1), 256, 0, st>>>(offsets, n_seqs, pre, starts);
    SM_LAUNCHED();
}

}  // namespace smb200
