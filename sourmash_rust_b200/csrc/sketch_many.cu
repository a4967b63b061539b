// sketch_many.cu -- one fresh sketch PER SEQUENCE of a batch, all in one pass: the sketching half of
// "sketch N genomes, then compare them all" (BASELINE configs 3 and 5), for up to six parameter sets at once.
//
// Equivalent reference loop (src/lib.rs:142-174, 252-305; src/index/linear.rs:47-50), one collection per template:
//     for s in sequences { for t in templates { let mut mh = KmerMinHash::new(t.num, t.ksize, t.is_protein, t.seed,
//                          t.max_hash, false); mh.add_sequence(s, /*force=*/true); collection[t].push(mh) } }
// Calling the per-object ABI N times pays a launch, a threshold read-back and a fold per genome -- for a
// 5 Mbp genome ten times the 28 us its k-mers take.  Here the sketch kernels (sketch.cu, protein.cu) run ONCE
// over the whole batch per template and report every surviving hash with its position; positions become
// sequence ids, two stable radix sorts (by hash, then by sequence) group them, and a flag / scan / compact
// pass drops duplicates, applies `num` per sequence and leaves the packed CSR of a SketchCollection.
//   scaled sketches (num = 0, max_hash > 0): the threshold is max_hash, exact by construction;
//   num sketches (num > 0, max_hash = 0): the kernel's threshold is an estimate from the median
//     sequence length (16 x num expected survivors); a sequence that ends up with fewer than `num`
//     distinct survivors under a threshold that was not "everything" is sketched again on its own
//     through the per-object path, so the result is exact for every input.
// Shared by the templates of one call: the host-to-device copy of the batch, the staging of each tile by the
// fused k = 21/31/51 kernel (DNA templates that fused_members groups), and the six-frame translation of the
// batch (protein templates; each hashes its own windows).  Per template: threshold, survivor buffer and
// counter, the overflow re-run, the grouping into rows and the redo of sequences cut short.
#include <algorithm>
#include <memory>
#include <vector>

#include "collection.hpp"
#include "kernels.cuh"

namespace smb200 {

namespace {

__global__ void __launch_bounds__(256) pos_to_seq_kernel(const uint64_t *pos /* may alias seq */, uint64_t n,
                                                         const uint64_t *__restrict__ starts, uint64_t n_seqs, uint64_t *seq) {
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        const uint64_t p = pos[i];
        uint64_t lo = 0, hi = n_seqs;  // largest s with starts[s] <= p
        while (hi - lo > 1) {
            const uint64_t mid = (lo + hi) >> 1;
            if (starts[mid] <= p) lo = mid; else hi = mid;
        }
        seq[i] = lo;
    }
}
// sorted by (seq, hash): flags[i] = first occurrence of its (seq, hash); seg_head[i] = first entry of its sequence
__global__ void __launch_bounds__(256) many_flags_kernel(const uint64_t *__restrict__ seq, const uint64_t *__restrict__ hash,
                                                         uint64_t n, uint64_t *flags) {
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride)
        flags[i] = (i == 0 || seq[i] != seq[i - 1] || hash[i] != hash[i - 1]) ? 1 : 0;
}
// seg_base[s] = number of distinct entries before the first entry of sequence s
__global__ void __launch_bounds__(256) many_seg_base_kernel(const uint64_t *__restrict__ seq, const uint64_t *__restrict__ pre,
                                                            uint64_t n, uint64_t *seg_base) {
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride)
        if (i == 0 || seq[i] != seq[i - 1]) seg_base[seq[i]] = pre[i];
}
// keep[i] = distinct and among the first `num` distinct hashes of its sequence (num = 0: all);
// distinct[s] / kept[s] count per sequence
__global__ void __launch_bounds__(256) many_keep_kernel(const uint64_t *__restrict__ seq, const uint64_t *__restrict__ flags,
                                                        const uint64_t *__restrict__ pre, const uint64_t *__restrict__ seg_base,
                                                        uint64_t n, uint32_t num, uint64_t *keep, unsigned long long *distinct,
                                                        unsigned long long *kept) {
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        uint64_t k = 0;
        if (flags[i]) {
            const uint64_t s = seq[i];
            atomicAdd(&distinct[s], 1ull);
            if (num == 0 || pre[i] - seg_base[s] < num) {
                k = 1;
                atomicAdd(&kept[s], 1ull);
            }
        }
        keep[i] = k;
    }
}
__global__ void __launch_bounds__(256) many_compact_kernel(const uint64_t *__restrict__ hash, const uint64_t *__restrict__ keep,
                                                           const uint64_t *__restrict__ kpre, uint64_t n, uint64_t *out) {
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride)
        if (keep[i]) out[kpre[i]] = hash[i];
}
constexpr int MAX_TEMPLATES = 6;
// control words of one call (device memory): per template a threshold and a survivor counter, and the tile
// counter pair that every sketch launch of the call shares (they are ordered on one stream)
enum { CTL_THR = 0, CTL_CNT = MAX_TEMPLATES, CTL_TILES = 2 * MAX_TEMPLATES, CTL_WORDS };
struct CtlInit {
    unsigned long long thr[MAX_TEMPLATES];
    int n;
};
__global__ void many_set_ctl_kernel(unsigned long long *ctl, const CtlInit init) {
#pragma unroll
    for (int m = 0; m < MAX_TEMPLATES; m++) {
        if (m < init.n) {
            ctl[CTL_THR + m] = init.thr[m];
            ctl[CTL_CNT + m] = 0;
        }
    }
    ctl[CTL_TILES] = 0;  // both u32 tile counters
}

constexpr uint64_t U64_MAX = ~0ull;
unsigned grid_for(uint64_t n) { return (unsigned)std::max<uint64_t>(1, std::min<uint64_t>((n + 255) / 256, 148 * 16)); }
int bits_of(uint64_t x) { int b = 0; while (x) { b++; x >>= 1; } return std::max(1, b); }

// One template's `count` survivors (hash, pos) -> the packed rows of c (c.h_offsets, c.d_hashes, c.n_hashes).
// seq_start[s] = position of the first window of sequence s, non-decreasing (DNA: the byte offsets; protein: the
// compacted residue index of its slot region).  h_distinct[s] receives the distinct survivors of sequence s.
void group_survivors(Context &ctx, uint64_t *hash, uint64_t *pos, uint64_t count, const uint64_t *seq_start, uint64_t thr,
                     uint32_t num, SketchCollection &c, std::vector<uint64_t> &h_distinct) {
    if (!count) return;
    cudaStream_t st = ctx.stream;
    const uint64_t n_seqs = c.n_rows;
    std::vector<uint64_t> h_kept(n_seqs, 0);
    // ---- positions -> sequence ids; group by (sequence, hash) ---------------------------------------
    uint64_t *seq = pos;
    pos_to_seq_kernel<<<grid_for(count), 256, 0, st>>>(pos, count, seq_start, n_seqs, seq);  // in place: pos -> seq
    SM_LAUNCHED();
    ctx.sort_tmp_k.reserve((count + 1) * 8);
    ctx.sort_tmp_v.reserve((count + 1) * 8);
    ctx.scan_tmp.reserve(std::max(radix_sort_scan_bytes(count), scan_tmp_bytes(std::max<uint64_t>(count, n_seqs + 1))) + 256);
    radix_sort_pairs(hash, seq, count, ctx.sort_tmp_k.as<uint64_t>(), ctx.sort_tmp_v.as<uint64_t>(), bits_of(thr), ctx.scan_tmp.p,
                     ctx.scan_tmp.cap, st);
    radix_sort_pairs(seq, hash, count, ctx.sort_tmp_k.as<uint64_t>(), ctx.sort_tmp_v.as<uint64_t>(), bits_of(n_seqs), ctx.scan_tmp.p,
                     ctx.scan_tmp.cap, st);
    // ---- distinct, first `num` per sequence, compact ---------------------------------------------------
    for (int i = 2; i < 6; i++) ctx.join[i].reserve((std::max(count, n_seqs) + 2) * 8);
    ctx.misc[0].reserve((n_seqs + 2) * 8);
    ctx.misc[1].reserve((n_seqs + 2) * 8);
    uint64_t *flags = ctx.join[2].as<uint64_t>(), *pre = ctx.join[3].as<uint64_t>(), *keep = ctx.join[4].as<uint64_t>();
    uint64_t *seg_base = ctx.join[5].as<uint64_t>();
    unsigned long long *distinct = ctx.misc[0].as<unsigned long long>(), *kept = ctx.misc[1].as<unsigned long long>();
    SM_CUDA(cudaMemsetAsync(seg_base, 0, (n_seqs + 1) * 8, st));
    SM_CUDA(cudaMemsetAsync(distinct, 0, (n_seqs + 1) * 8, st));
    SM_CUDA(cudaMemsetAsync(kept, 0, (n_seqs + 1) * 8, st));
    many_flags_kernel<<<grid_for(count), 256, 0, st>>>(seq, hash, count, flags);
    SM_LAUNCHED();
    scan_exclusive_u64(flags, pre, count, ctx.scan_tmp.p, st);
    many_seg_base_kernel<<<grid_for(count), 256, 0, st>>>(seq, pre, count, seg_base);
    SM_LAUNCHED();
    many_keep_kernel<<<grid_for(count), 256, 0, st>>>(seq, flags, pre, seg_base, count, num, keep, distinct, kept);
    SM_LAUNCHED();
    scan_exclusive_u64(keep, pre, count, ctx.scan_tmp.p, st);  // pre now: output slot of every kept entry
    SM_CUDA(cudaMemcpyAsync(h_distinct.data(), distinct, n_seqs * 8, cudaMemcpyDeviceToHost, st));
    SM_CUDA(cudaMemcpyAsync(h_kept.data(), kept, n_seqs * 8, cudaMemcpyDeviceToHost, st));
    ctx.sync();
    uint64_t total = 0;
    for (uint64_t s = 0; s < n_seqs; s++) { c.h_offsets[s] = total; total += h_kept[s]; }
    c.h_offsets[n_seqs] = total;
    c.d_hashes.reserve((total + 4) * 8);
    many_compact_kernel<<<grid_for(count), 256, 0, st>>>(hash, keep, pre, count, c.d_hashes.as<uint64_t>());
    SM_LAUNCHED();
    c.n_hashes = total;
}

// num sketches: the sequences that kept fewer than `num` distinct survivors under an estimated threshold are sketched
// again on their own through the per-object path and patched in on the host (rare, and those sequences are short by
// construction)
void redo_short(Context &ctx, SketchCollection &c, const SketchParams &p, const uint8_t *buf, const std::vector<uint64_t> &h_off,
                bool on_device, const std::vector<uint64_t> &h_distinct) {
    cudaStream_t st = ctx.stream;
    const uint64_t n_seqs = c.n_rows;
    std::vector<uint64_t> redo;
    for (uint64_t s = 0; s < n_seqs; s++)
        if (h_distinct[s] < p.num) redo.push_back(s);
    if (redo.empty()) return;
    std::vector<uint64_t> h_hashes(c.n_hashes);
    if (c.n_hashes) SM_CUDA(cudaMemcpyAsync(h_hashes.data(), c.d_hashes.p, c.n_hashes * 8, cudaMemcpyDeviceToHost, st));
    ctx.sync();
    std::vector<std::vector<uint64_t>> fixed(redo.size());
    std::vector<uint8_t> tmp;
    for (size_t r = 0; r < redo.size(); r++) {
        const uint64_t s = redo[r], len = h_off[s + 1] - h_off[s];
        KmerMinHash mh(p.num, p.ksize, p.is_protein, p.seed, 0, false);
        if (len) {
            tmp.resize(len);
            if (on_device) {
                SM_CUDA(cudaMemcpyAsync(tmp.data(), buf + h_off[s], len, cudaMemcpyDeviceToHost, st));
                ctx.sync();
            } else {
                std::copy(buf + h_off[s], buf + h_off[s] + len, tmp.begin());
            }
            mh.add_sequence(tmp.data(), len, true);
        }
        fixed[r] = mh.mins();
    }
    std::vector<uint64_t> out_h, out_o(n_seqs + 1, 0);
    size_t r = 0;
    for (uint64_t s = 0; s < n_seqs; s++) {
        out_o[s] = out_h.size();
        if (r < redo.size() && redo[r] == s) {
            out_h.insert(out_h.end(), fixed[r].begin(), fixed[r].end());
            r++;
        } else {
            out_h.insert(out_h.end(), h_hashes.begin() + c.h_offsets[s], h_hashes.begin() + c.h_offsets[s + 1]);
        }
    }
    out_o[n_seqs] = out_h.size();
    c.h_offsets = out_o;
    c.n_hashes = out_h.size();
    c.d_hashes.reserve((c.n_hashes + 4) * 8);
    if (c.n_hashes) SM_CUDA(cudaMemcpyAsync(c.d_hashes.p, out_h.data(), c.n_hashes * 8, cudaMemcpyHostToDevice, st));
    ctx.sync();
}

}  // namespace

std::vector<std::unique_ptr<SketchCollection>> sketch_collections(const uint8_t *buf, const uint64_t *offsets, uint64_t n_seqs,
                                                                  const std::vector<SketchParams> &ps, bool on_device) {
    const int nt = (int)ps.size();
    if (nt < 1 || nt > MAX_TEMPLATES) throw_internal("sketch_collections takes 1 to 6 templates");
    for (const SketchParams &p : ps) {
        if ((p.num == 0) == (p.max_hash == 0))
            throw_internal("sketch_collection takes either num > 0 (bottom-num sketches) or max_hash > 0 (scaled sketches)");
        if (p.ksize == 0) throw_internal("ksize 0");
        if (p.is_protein && p.ksize < 3)  // as add_sequences: the reference reaches slice::windows(0), which panics
            throw SourmashError(ERR_PANIC, "sourmash panicked: size is zero");
    }
    Context &ctx = Context::get();
    cudaStream_t st = ctx.stream;
    std::vector<std::unique_ptr<SketchCollection>> cs(nt);
    for (int m = 0; m < nt; m++) {
        cs[m].reset(new SketchCollection());
        SketchCollection &c = *cs[m];
        c.have_params = true;
        c.ksize = ps[m].ksize; c.seed = ps[m].seed; c.max_hash = ps[m].max_hash; c.is_protein = ps[m].is_protein;
        c.n_rows = n_seqs;
        c.h_nums.assign(n_seqs, ps[m].num);
        c.h_offsets.assign(n_seqs + 1, 0);
    }
    if (n_seqs == 0) return cs;

    // ---- the batch and its offsets on the device, once for every template ------------------------------
    std::vector<uint64_t> h_off(n_seqs + 1);
    if (on_device) {
        SM_CUDA(cudaMemcpyAsync(h_off.data(), offsets, (n_seqs + 1) * 8, cudaMemcpyDeviceToHost, st));
        ctx.sync();
    } else {
        std::copy(offsets, offsets + n_seqs + 1, h_off.begin());
    }
    if (h_off[0] != 0) throw_internal("offsets[0] must be 0");
    for (uint64_t s = 0; s < n_seqs; s++)
        if (h_off[s + 1] < h_off[s]) throw_internal("offsets must be non-decreasing");
    const uint64_t n = h_off[n_seqs];
    for (const SketchParams &p : ps)
        if (n && !p.is_protein && p.ksize > (uint32_t)SK_MAX_GENERIC_K)
            throw_internal("ksize above 8192 is not supported by the GPU sketcher");
    const uint8_t *d_buf = buf;
    const uint64_t *d_off = offsets;
    if (!on_device) {
        ctx.ascii.reserve(((n + 15) & ~15ull) + 256);
        ctx.offsets.reserve((n_seqs + 1) * 8);
        if (n) SM_CUDA(cudaMemcpyAsync(ctx.ascii.p, buf, n, cudaMemcpyHostToDevice, st));
        SM_CUDA(cudaMemcpyAsync(ctx.offsets.p, h_off.data(), (n_seqs + 1) * 8, cudaMemcpyHostToDevice, st));
        d_buf = ctx.ascii.as<uint8_t>();
        d_off = ctx.offsets.as<uint64_t>();
    } else if ((reinterpret_cast<uintptr_t>(buf) & 15) != 0) {
        throw_internal("device sequence buffer must be 16-byte aligned");
    }

    // ---- per template: threshold and a survivor region [base, base + cap) of the shared buffers -----------
    // windows per sequence: about len for DNA, about 2 len for protein (six frames of len / 3 residues)
    const uint64_t protein_windows = protein_slots(n, n_seqs);
    double median = 1.0;
    if (std::any_of(ps.begin(), ps.end(), [](const SketchParams &p) { return p.max_hash == 0; })) {
        std::vector<uint64_t> lens(n_seqs);
        for (uint64_t s = 0; s < n_seqs; s++) lens[s] = h_off[s + 1] - h_off[s];
        std::nth_element(lens.begin(), lens.begin() + n_seqs / 2, lens.end());
        median = (double)std::max<uint64_t>(1, lens[n_seqs / 2]);
    }
    std::vector<uint64_t> thr(nt), cap(nt), base(nt), count(nt, 0);
    uint64_t total = 0;
    for (int m = 0; m < nt; m++) {
        const SketchParams &p = ps[m];
        double frac = 1.0;
        thr[m] = U64_MAX;
        if (p.max_hash) {
            thr[m] = p.max_hash;
            frac = (double)p.max_hash / 18446744073709551616.0;
        } else {
            frac = std::min(1.0, 16.0 * (double)p.num / (p.is_protein ? 2.0 * median : median));
            if (frac < 1.0) thr[m] = (uint64_t)(frac * 18446744073709551616.0);
        }
        cap[m] = (uint64_t)(frac * 1.25 * (double)(p.is_protein ? protein_windows : n)) + 4096;
        base[m] = total;
        total += cap[m];
    }
    ctx.join[0].reserve((total + 1) * 8);
    ctx.join[1].reserve((total + 1) * 8);
    ctx.misc[6].reserve(CTL_WORDS * 8);
    unsigned long long *ctl = ctx.misc[6].as<unsigned long long>();

    // ---- protein templates: one translation of the batch (protein.cu), at the smallest protein ksize --------
    ProteinBatch pb;
    pb.buf = d_buf; pb.n = n; pb.offsets = d_off; pb.n_seqs = n_seqs; pb.read_len = 0; pb.ksize = 0; pb.seed = 0;
    for (const SketchParams &p : ps)
        if (p.is_protein) pb.ksize = pb.ksize ? std::min(pb.ksize, p.ksize) : p.ksize;
    uint8_t *aa = nullptr, *comp = nullptr;
    uint64_t *pflags = nullptr, *ppre = nullptr, *pstarts = nullptr;
    if (pb.ksize && n) {
        ctx.misc[0].reserve(protein_windows + 64);
        ctx.misc[1].reserve(protein_windows + 64);
        ctx.misc[2].reserve((protein_windows + 2) * 8);
        ctx.misc[3].reserve((protein_windows + 2) * 8);
        ctx.misc[4].reserve((n_seqs + 1) * 8);
        ctx.scan_tmp.reserve(scan_tmp_bytes(protein_windows + 1) + 256);
        aa = ctx.misc[0].as<uint8_t>(); comp = ctx.misc[1].as<uint8_t>();
        pflags = ctx.misc[2].as<uint64_t>(); ppre = ctx.misc[3].as<uint64_t>(); pstarts = ctx.misc[4].as<uint64_t>();
        launch_protein_translate(pb, aa, comp, pflags, ppre, ctx.scan_tmp.p, st);
        launch_protein_seq_starts(d_off, n_seqs, ppre, pstarts, st);
    }

    // ---- sketch kernels over the whole batch: survivors (hash, position) per template ---------------------
    auto out_of = [&](int m) {
        SketchOut o;
        o.thr = reinterpret_cast<const uint64_t *>(ctl + CTL_THR + m);
        o.hash = ctx.join[0].as<uint64_t>() + base[m];
        o.pos = ctx.join[1].as<uint64_t>() + base[m];
        o.cap = cap[m];
        o.counter = ctl + CTL_CNT + m;
        return o;
    };
    auto batch_of = [&](uint64_t seed) {
        SketchBatch sb;
        sb.buf = d_buf; sb.n = n; sb.n_limit = n; sb.offsets = d_off; sb.n_seqs = n_seqs; sb.read_len = 0; sb.tile_lo = 0;
        sb.seed = seed; sb.pos_base = 0; sb.first_bad = nullptr;  // force = true: invalid k-mers are skipped
        sb.tile_ctr = reinterpret_cast<uint32_t *>(ctl + CTL_TILES);
        return sb;
    };
    // the launches of templates `which` (ascending): the DNA templates fused_members picks share one launch
    auto launch = [&](const std::vector<int> &which) {
        std::vector<SketchParams> sub;
        for (int m : which) sub.push_back(ps[m]);
        const std::vector<int> fused = fused_members(sub);
        if (!fused.empty()) {
            uint32_t ks[3];
            SketchOuts outs;
            for (size_t j = 0; j < 3; j++) {
                const int m = which[fused[std::min(j, fused.size() - 1)]];
                outs.o[j] = out_of(m);
                outs.first_bad[j] = nullptr;
                if (j < fused.size()) ks[j] = ps[m].ksize;
            }
            launch_sketch_multi(ks, (int)fused.size(), batch_of(sub[fused[0]].seed), outs, sketch_tile_count(n, n), ctx.sm_count, st);
        }
        for (size_t i = 0; i < which.size(); i++) {
            if (std::find(fused.begin(), fused.end(), (int)i) != fused.end()) continue;
            const int m = which[i];
            if (ps[m].is_protein) {
                ProteinBatch q = pb;
                q.ksize = ps[m].ksize;
                q.seed = ps[m].seed;
                launch_protein_hash(q, out_of(m), comp, pflags, ppre, st);
            } else {
                launch_sketch(ps[m].ksize, batch_of(ps[m].seed), out_of(m), sketch_tile_count(n, n), ctx.sm_count, st);
            }
        }
    };
    std::vector<int> which(nt);
    for (int m = 0; m < nt; m++) which[m] = m;
    std::vector<uint64_t> h_count(nt);
    for (int attempt = 0;; attempt++) {
        if (attempt > 8) throw_internal("sketch_collection: survivor buffer did not converge");
        CtlInit init;
        init.n = nt;
        for (int m = 0; m < nt; m++) init.thr[m] = thr[m];
        many_set_ctl_kernel<<<1, 1, 0, st>>>(ctl, init);
        SM_LAUNCHED();
        if (n) launch(which);
        SM_CUDA(cudaMemcpyAsync(h_count.data(), ctl + CTL_CNT, nt * 8, cudaMemcpyDeviceToHost, st));
        ctx.sync();
        std::vector<int> over;
        for (int m : which) {
            count[m] = h_count[m];
            if (count[m] > cap[m]) over.push_back(m);
        }
        if (over.empty()) break;
        // entries beyond cap were dropped but counted: run those templates again, each in a new region with room for
        // all; the other templates' survivors stay where they are (unless every template runs again)
        const bool all = over.size() == (size_t)nt;
        const uint64_t kept_bytes = all ? 0 : total * 8;
        if (all) total = 0;
        for (int m : over) {
            cap[m] = count[m] + 4096;
            base[m] = total;
            total += cap[m];
        }
        ctx.join[0].reserve((total + 1) * 8, st, !all, kept_bytes);
        ctx.join[1].reserve((total + 1) * 8, st, !all, kept_bytes);
        which = over;
    }

    // ---- per template: survivors -> rows; num sketches: sequences cut short again on their own; upload ------
    std::vector<std::vector<uint64_t>> distinct(nt, std::vector<uint64_t>(n_seqs, 0));
    for (int m = 0; m < nt; m++)
        group_survivors(ctx, ctx.join[0].as<uint64_t>() + base[m], ctx.join[1].as<uint64_t>() + base[m], count[m],
                        ps[m].is_protein ? pstarts : d_off, thr[m], ps[m].num, *cs[m], distinct[m]);
    for (int m = 0; m < nt; m++)
        if (ps[m].num && thr[m] != U64_MAX) redo_short(ctx, *cs[m], ps[m], buf, h_off, on_device, distinct[m]);
    for (int m = 0; m < nt; m++) {
        SketchCollection &c = *cs[m];
        c.d_offsets.reserve((n_seqs + 1) * 8);
        c.d_nums.reserve((n_seqs + 1) * 4);
        SM_CUDA(cudaMemcpyAsync(c.d_offsets.p, c.h_offsets.data(), (n_seqs + 1) * 8, cudaMemcpyHostToDevice, st));
        SM_CUDA(cudaMemcpyAsync(c.d_nums.p, c.h_nums.data(), n_seqs * 4, cudaMemcpyHostToDevice, st));
        c.max_len = 0;
        for (uint64_t s = 0; s < n_seqs; s++) c.max_len = std::max<uint32_t>(c.max_len, (uint32_t)(c.h_offsets[s + 1] - c.h_offsets[s]));
    }
    ctx.sync();
    return cs;
}

SketchCollection *sketch_collection(const uint8_t *buf, const uint64_t *offsets, uint64_t n_seqs, uint32_t num, uint32_t ksize,
                                    uint64_t seed, uint64_t max_hash, bool on_device) {
    return sketch_collections(buf, offsets, n_seqs, {SketchParams{num, ksize, false, seed, max_hash}}, on_device)[0].release();
}

}  // namespace smb200
