// comm.cu -- the multi-GPU exchange steps of the path, inside the library, over NCCL (NVLink 5 / NVSwitch).
//
// One process per GPU.  The reference has no distributed code (SURVEY 5); what shards is algebra (SURVEY 8(e)):
//   * sketches of disjoint read sets combine by KmerMinHash::merge (lib.rs:307-403)          -> comm_allmerge
//   * the rows of the all-vs-all matrix are independent, every rank needs all columns        -> collection_allgather,
//                                                                                               compare_matrix_allgather
//   * LinearIndex::find over a partitioned index = concatenation of the parts' hit lists
//     in partition order (linear.rs:34-44)                                                    -> linear_find_sharded
//
// NCCL is bound at run time (dlopen of libnccl.so.2 -- the copy already in the process when the host program
// has one, e.g. PyTorch's): the library has no link-time dependency on it, and a single-GPU user never loads it.
// The unique id travels by whatever channel the host program has (MPI, a file, torch.distributed): the library
// opens no sockets of its own.
#include "comm.hpp"

#include <dlfcn.h>
#include <nccl.h>

#include <algorithm>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <mutex>

#include "kernels.cuh"

namespace smb200 {

namespace {

struct NcclApi {
    void *handle = nullptr;
    ncclResult_t (*GetUniqueId)(ncclUniqueId *) = nullptr;
    ncclResult_t (*CommInitRank)(ncclComm_t *, int, ncclUniqueId, int) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    ncclResult_t (*AllGather)(const void *, void *, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*Send)(const void *, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*Recv)(void *, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*GroupStart)() = nullptr;
    ncclResult_t (*GroupEnd)() = nullptr;
    const char *(*GetErrorString)(ncclResult_t) = nullptr;
    ncclResult_t (*GetVersion)(int *) = nullptr;
};
NcclApi g_nccl;

struct Comm {
    ncclComm_t comm = nullptr;
    int rank = 0, world = 1;
    cudaStream_t stream = nullptr;            // collectives run here, beside the calling thread's compute stream
    cudaEvent_t ev_ready = nullptr, ev_done = nullptr;
    cudaStream_t build_stream = nullptr;      // the join table of a rank's own rows is built here, beside the exchange
    cudaEvent_t ev_build_go = nullptr, ev_build_done = nullptr;
    unsigned long long *d_hdr = nullptr;      // [HDR] mine + [world * HDR] everybody's
    unsigned long long *h_hdr = nullptr;      // pinned mirror of the gathered part
};
Comm g_comm;
std::mutex g_comm_mutex;  // one collective at a time per process (NCCL's own rule for one communicator)

constexpr int HDR = 8;  // u64 per rank: n_rows, n_hashes, max_len, ksize, seed, max_hash, is_protein | have_params << 1, spare

#define SM_NCCL(expr)                                                                                       \
    do {                                                                                                    \
        ncclResult_t _r = (expr);                                                                           \
        if (_r != ncclSuccess)                                                                              \
            throw_internal(std::string("NCCL: ") + (g_nccl.GetErrorString ? g_nccl.GetErrorString(_r) : "error") + \
                           " at " + __FILE__ + ":" + std::to_string(__LINE__) + " (" #expr ")");          \
    } while (0)

void load_nccl() {
    if (g_nccl.handle) return;
    void *h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_NOLOAD);  // the host program's copy, if it has one
    if (!h) h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
    if (!h) h = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
    if (!h) throw_internal(std::string("multi-GPU entry points need NCCL (libnccl.so.2): ") + dlerror());
    auto sym = [&](const char *name) {
        void *p = dlsym(h, name);
        if (!p) throw_internal(std::string("libnccl.so.2 lacks ") + name);
        return p;
    };
    g_nccl.GetUniqueId = reinterpret_cast<decltype(g_nccl.GetUniqueId)>(sym("ncclGetUniqueId"));
    g_nccl.CommInitRank = reinterpret_cast<decltype(g_nccl.CommInitRank)>(sym("ncclCommInitRank"));
    g_nccl.CommDestroy = reinterpret_cast<decltype(g_nccl.CommDestroy)>(sym("ncclCommDestroy"));
    g_nccl.AllGather = reinterpret_cast<decltype(g_nccl.AllGather)>(sym("ncclAllGather"));
    g_nccl.Send = reinterpret_cast<decltype(g_nccl.Send)>(sym("ncclSend"));
    g_nccl.Recv = reinterpret_cast<decltype(g_nccl.Recv)>(sym("ncclRecv"));
    g_nccl.GroupStart = reinterpret_cast<decltype(g_nccl.GroupStart)>(sym("ncclGroupStart"));
    g_nccl.GroupEnd = reinterpret_cast<decltype(g_nccl.GroupEnd)>(sym("ncclGroupEnd"));
    g_nccl.GetErrorString = reinterpret_cast<decltype(g_nccl.GetErrorString)>(sym("ncclGetErrorString"));
    g_nccl.GetVersion = reinterpret_cast<decltype(g_nccl.GetVersion)>(sym("ncclGetVersion"));
    g_nccl.handle = h;
}

__global__ void put_header_kernel(unsigned long long *dst, unsigned long long a, unsigned long long b, unsigned long long c,
                                  unsigned long long d, unsigned long long e, unsigned long long f, unsigned long long g,
                                  unsigned long long h) {
    dst[0] = a; dst[1] = b; dst[2] = c; dst[3] = d; dst[4] = e; dst[5] = f; dst[6] = g; dst[7] = h;
}
__global__ void words_to_host_kernel(const unsigned long long *src, unsigned long long *dst, int n) {
    for (int i = threadIdx.x; i < n; i += blockDim.x) dst[i] = src[i];
}
// hits[i] += base for a rank's local row ids
__global__ void add_base_kernel(uint64_t *__restrict__ v, uint64_t n, uint64_t base) {
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) v[i] += base;
}

// every rank's 8-word header, on the host (one small all-gather + one kernel store into pinned memory: the only
// host round trip of an exchange whose sizes are not known in advance)
// (in two halves: what the caller queues between them runs while the headers are on their way)
void exchange_headers_begin(const unsigned long long mine[HDR]) {
    Comm &c = g_comm;
    put_header_kernel<<<1, 1, 0, c.stream>>>(c.d_hdr, mine[0], mine[1], mine[2], mine[3], mine[4], mine[5], mine[6], mine[7]);
    SM_LAUNCHED();
    SM_NCCL(g_nccl.AllGather(c.d_hdr, c.d_hdr + HDR, HDR, ncclUint64, c.comm, c.stream));
    words_to_host_kernel<<<1, 64, 0, c.stream>>>(c.d_hdr + HDR, c.h_hdr, c.world * HDR);
    SM_LAUNCHED();
}
void exchange_headers_finish() { SM_CUDA(cudaStreamSynchronize(g_comm.stream)); }
void exchange_headers(const unsigned long long mine[HDR]) {
    exchange_headers_begin(mine);
    exchange_headers_finish();
}

// variable-size all-gather: rank r's `count[r]` elements land at recv + base[r].  Equal counts (fixed-width `num`
// sketches, the usual case): one ncclAllGather.  Otherwise point-to-point sends and receives, which NCCL fuses into one
// kernel inside a group (called between GroupStart / GroupEnd); the rank's own part is a device copy.
void allgatherv(const void *send, void *recv, const std::vector<uint64_t> &count, const std::vector<uint64_t> &base,
                size_t elem_bytes, ncclDataType_t type) {
    Comm &c = g_comm;
    bool equal = true;
    for (int r = 0; r < c.world; r++) equal = equal && count[r] == count[0] && base[r] == (uint64_t)r * count[0];
    if (equal) {
        if (count[0]) SM_NCCL(g_nccl.AllGather(send, recv, count[0], type, c.comm, c.stream));
        return;
    }
    for (int r = 0; r < c.world; r++) {
        if (r == c.rank) {
            if (count[r])
                SM_CUDA(cudaMemcpyAsync(static_cast<char *>(recv) + base[r] * elem_bytes, send, count[r] * elem_bytes,
                                        cudaMemcpyDeviceToDevice, c.stream));
            continue;
        }
        if (count[c.rank]) SM_NCCL(g_nccl.Send(send, count[c.rank], type, r, c.comm, c.stream));
        if (count[r]) SM_NCCL(g_nccl.Recv(static_cast<char *>(recv) + base[r] * elem_bytes, count[r], type, r, c.comm, c.stream));
    }
}

// [len, num] per row -> len as u64 (for the scan into offsets) and num
__global__ void unpack_rowinfo_kernel(const uint2 *__restrict__ info, uint64_t n, uint64_t *__restrict__ lens, uint32_t *__restrict__ nums) {
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        const uint2 v = info[i];
        lens[i] = v.x;
        nums[i] = v.y;
    }
}
// offsets[i] = i * len (i <= n), nums[i] = num
__global__ void uniform_rows_kernel(uint64_t *__restrict__ offsets, uint32_t *__restrict__ nums, uint64_t n, uint64_t len, uint32_t num) {
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i <= n; i += stride) {
        offsets[i] = i * len;
        if (i < n) nums[i] = num;
    }
}
// [len, num] of the local rows
__global__ void pack_rowinfo_kernel(const uint64_t *__restrict__ offsets, const uint32_t *__restrict__ nums, uint64_t n, uint2 *__restrict__ info) {
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride)
        info[i] = make_uint2((uint32_t)(offsets[i + 1] - offsets[i]), nums[i]);
}

}  // namespace

// ---------------------------------------------------------------------------------------------------------
void comm_unique_id(uint8_t out[COMM_ID_BYTES]) {
    load_nccl();
    static_assert(sizeof(ncclUniqueId) == COMM_ID_BYTES, "ncclUniqueId size");
    ncclUniqueId id;
    SM_NCCL(g_nccl.GetUniqueId(&id));
    memcpy(out, &id, COMM_ID_BYTES);
}

void comm_init(const uint8_t id_bytes[COMM_ID_BYTES], int rank, int world) {
    std::lock_guard<std::mutex> lk(g_comm_mutex);
    if (g_comm.comm) throw_internal("communicator already initialised");
    if (world < 1 || rank < 0 || rank >= world) throw_internal("bad rank / world size");
    load_nccl();
    Context &ctx = Context::get();  // binds the process's device first
    (void)ctx;
    ncclUniqueId id;
    memcpy(&id, id_bytes, COMM_ID_BYTES);
    Comm c;
    c.rank = rank;
    c.world = world;
    SM_NCCL(g_nccl.CommInitRank(&c.comm, world, id, rank));
    // the collectives' stream has the greatest priority: NCCL's few CTAs are placed ahead of the queued CTAs of a
    // GPU-filling table build or probe on the compute streams instead of waiting for those kernels to drain
    int prio_least = 0, prio_greatest = 0;
    SM_CUDA(cudaDeviceGetStreamPriorityRange(&prio_least, &prio_greatest));
    SM_CUDA(cudaStreamCreateWithPriority(&c.stream, cudaStreamNonBlocking, prio_greatest));
    SM_CUDA(cudaEventCreateWithFlags(&c.ev_ready, cudaEventDisableTiming));
    SM_CUDA(cudaEventCreateWithFlags(&c.ev_done, cudaEventDisableTiming));
    SM_CUDA(cudaStreamCreateWithFlags(&c.build_stream, cudaStreamNonBlocking));
    SM_CUDA(cudaEventCreateWithFlags(&c.ev_build_go, cudaEventDisableTiming));
    SM_CUDA(cudaEventCreateWithFlags(&c.ev_build_done, cudaEventDisableTiming));
    SM_CUDA(cudaMalloc(&c.d_hdr, (size_t)(world + 1) * HDR * 8));
    SM_CUDA(cudaMallocHost(&c.h_hdr, (size_t)world * HDR * 8));
    g_comm = c;
    // first collective here, not inside somebody's timed exchange: NCCL sets its channels up lazily
    unsigned long long zero[HDR] = {0};
    exchange_headers(zero);
}

void comm_destroy() {
    std::lock_guard<std::mutex> lk(g_comm_mutex);
    if (!g_comm.comm) return;
    cudaStreamSynchronize(g_comm.stream);
    g_nccl.CommDestroy(g_comm.comm);
    cudaStreamDestroy(g_comm.stream);
    cudaEventDestroy(g_comm.ev_ready);
    cudaEventDestroy(g_comm.ev_done);
    cudaStreamSynchronize(g_comm.build_stream);
    cudaStreamDestroy(g_comm.build_stream);
    cudaEventDestroy(g_comm.ev_build_go);
    cudaEventDestroy(g_comm.ev_build_done);
    cudaFree(g_comm.d_hdr);
    cudaFreeHost(g_comm.h_hdr);
    g_comm = Comm();
}

int comm_rank() { return g_comm.comm ? g_comm.rank : 0; }
int comm_world() { return g_comm.comm ? g_comm.world : 1; }
int comm_nccl_version() {
    load_nccl();
    int v = 0;
    g_nccl.GetVersion(&v);
    return v;
}

// ---------------------------------------------------------------------------------------------------------
// all-gather of a packed collection.  `meanwhile` (optional) is called once the header exchange has been queued and
// before this thread waits for it: what it queues needs local data only and runs beside the exchange.
// ---------------------------------------------------------------------------------------------------------
// `hashes_ready` (optional, set non-null only for uniform rows on more than one rank): the compute stream is NOT made to
// wait for the hashes; the caller waits for that event before it touches them.
static SketchCollection *allgather_impl(SketchCollection &local, const std::function<void()> &meanwhile,
                                        cudaEvent_t *hashes_ready = nullptr) {
    if (hashes_ready) *hashes_ready = nullptr;
    Comm &c = g_comm;
    Context &ctx = Context::get();
    local.finalize();  // (rows were checked strictly ascending when the local collection was made: peers do the same)
    if (!c.comm) {
        // no communicator = a world of one: the gathered collection is a copy of the local one (NCCL is not loaded)
        std::unique_ptr<SketchCollection> out(new SketchCollection());
        ctx.adopt(out->owner);
        out->have_params = local.have_params;
        out->ksize = local.ksize; out->is_protein = local.is_protein; out->seed = local.seed; out->max_hash = local.max_hash;
        out->n_rows = local.n_rows; out->n_hashes = local.n_hashes; out->max_len = local.max_len;
        out->h_offsets.assign(local.h_offsets.begin(), local.h_offsets.begin() + local.n_rows + 1);
        out->h_nums.assign(local.h_nums.begin(), local.h_nums.begin() + local.n_rows);
        out->d_hashes.reserve((local.n_hashes + 4) * 8);
        out->d_offsets.reserve((local.n_rows + 2) * 8);
        out->d_nums.reserve((local.n_rows + 1) * 4);
        if (local.n_hashes) SM_CUDA(cudaMemcpyAsync(out->d_hashes.p, local.d_hashes.p, local.n_hashes * 8, cudaMemcpyDeviceToDevice, ctx.stream));
        SM_CUDA(cudaMemcpyAsync(out->d_offsets.p, local.d_offsets.p, (local.n_rows + 1) * 8, cudaMemcpyDeviceToDevice, ctx.stream));
        if (local.n_rows) SM_CUDA(cudaMemcpyAsync(out->d_nums.p, local.d_nums.p, local.n_rows * 4, cudaMemcpyDeviceToDevice, ctx.stream));
        if (meanwhile) meanwhile();
        out->dirty = false;
        return out.release();
    }
    // rows all of one length and one num (a collection of full `num` sketches): said in the header, so that the
    // receivers know every offset without seeing the row lengths
    bool uniform = local.n_rows > 0 && local.max_len < (1u << 31);
    const uint64_t len0 = local.n_rows ? local.h_offsets[1] - local.h_offsets[0] : 0;
    for (uint64_t i = 0; uniform && i < local.n_rows; i++)
        uniform = local.h_offsets[i + 1] - local.h_offsets[i] == len0 && local.h_nums[i] == local.h_nums[0];
    const unsigned long long shape = uniform ? ((1ull << 63) | (len0 << 32) | local.h_nums[0]) : 0;
    unsigned long long mine[HDR] = {local.n_rows, local.n_hashes, local.max_len, local.ksize, local.seed, local.max_hash,
                                    (unsigned long long)local.is_protein | ((unsigned long long)local.have_params << 1), shape};
    exchange_headers_begin(mine);
    if (meanwhile) meanwhile();
    exchange_headers_finish();
    const int W = c.world;
    std::vector<uint64_t> rows(W), hashes(W), row_base(W), hash_base(W);
    uint64_t n_rows = 0, n_hashes = 0, max_len = 0;
    unsigned long long all_shape = 0;   // the one shape every non-empty rank reported, or 1 = not uniform
    std::unique_ptr<SketchCollection> out(new SketchCollection());
    for (int r = 0; r < W; r++) {
        const unsigned long long *h = c.h_hdr + (size_t)r * HDR;
        if (h[0]) all_shape = (all_shape == 0 || all_shape == h[7]) && (h[7] >> 63) ? h[7] : 1;
        rows[r] = h[0]; hashes[r] = h[1];
        row_base[r] = n_rows; hash_base[r] = n_hashes;
        n_rows += h[0]; n_hashes += h[1];
        max_len = std::max<uint64_t>(max_len, h[2]);
        if (!(h[6] >> 1)) continue;  // an empty collection carries no parameters
        if (!out->have_params) {
            out->have_params = true;
            out->ksize = (uint32_t)h[3]; out->seed = h[4]; out->max_hash = h[5]; out->is_protein = h[6] & 1;
        } else {  // KmerMinHash::check_compatible across ranks (lib.rs:176-190), same order of tests
            if (out->ksize != (uint32_t)h[3]) throw SourmashError(ERR_MISMATCH_KSIZES, "different ksizes cannot be compared");
            if (out->is_protein != (bool)(h[6] & 1)) throw SourmashError(ERR_MISMATCH_DNAPROT, "DNA/prot minhashes cannot be compared");
            if (out->max_hash != h[5]) throw SourmashError(ERR_MISMATCH_MAXHASH, "mismatch in max_hash; comparison fail");
            if (out->seed != h[4]) throw SourmashError(ERR_MISMATCH_SEED, "mismatch in seed; comparison fail");
        }
    }
    ctx.adopt(out->owner);
    out->n_rows = n_rows;
    out->n_hashes = n_hashes;
    out->max_len = (uint32_t)max_len;
    out->d_hashes.reserve((n_hashes + 4) * 8);
    out->d_offsets.reserve((n_rows + 2) * 8);
    out->d_nums.reserve((n_rows + 1) * 4);
    const bool all_uniform = (all_shape >> 63) != 0;
    if (all_uniform) {
        // every row of every rank has the same length and num: only the hashes travel; offsets are i * length
        const uint64_t len = (all_shape >> 32) & 0x7FFFFFFFull;
        const uint32_t num = (uint32_t)all_shape;
        SM_CUDA(cudaEventRecord(c.ev_ready, ctx.stream));       // the output buffer is allocated (stream-ordered)
        SM_CUDA(cudaStreamWaitEvent(c.stream, c.ev_ready, 0));
        const bool deferred = hashes_ready && W > 1;      // the caller waits
        SM_NCCL(g_nccl.GroupStart());
        allgatherv(local.d_hashes.p, out->d_hashes.p, hashes, hash_base, 8, ncclUint64);
        SM_NCCL(g_nccl.GroupEnd());
        SM_CUDA(cudaEventRecord(c.ev_done, c.stream));
        if (deferred) *hashes_ready = c.ev_done;
        uniform_rows_kernel<<<(unsigned)std::min<uint64_t>((n_rows + 256) / 256, 148 * 8), 256, 0, ctx.stream>>>(
            out->d_offsets.as<uint64_t>(), out->d_nums.as<uint32_t>(), n_rows, len, num);
        SM_LAUNCHED();
        if (!deferred) SM_CUDA(cudaStreamWaitEvent(ctx.stream, c.ev_done, 0));
        out->h_offsets.resize(n_rows + 1);
        for (uint64_t i = 0; i <= n_rows; i++) out->h_offsets[i] = i * len;
        out->h_nums.assign(n_rows, num);
        if (out->h_offsets[n_rows] != n_hashes) throw_internal("all-gather: row lengths and hash counts disagree");
        out->dirty = false;
        return out.release();   // (nothing waits for the transfer here: the compare kernels are queued behind it)
    }
    // per row, [length, num] travel as one 8-byte record; on arrival the lengths are scanned into offsets.  This
    // thread's scratch: misc[0] = my records, misc[3] = everybody's, misc[2] = lengths as u64 (n_rows + 1 entries, the
    // last one zero: its exclusive scan = offsets), join[5] = scan scratch -- not misc[1], scan_tmp, sort_tmp_* or
    // join[0,1,6,7], which the table build that overlaps the transfer uses
    ctx.misc[0].reserve((local.n_rows + 1) * 8);
    ctx.misc[3].reserve((n_rows + 1) * 8);
    ctx.misc[2].reserve((n_rows + 2) * 8);
    uint2 *my_info = ctx.misc[0].as<uint2>(), *all_info = ctx.misc[3].as<uint2>();
    uint64_t *all_lens = ctx.misc[2].as<uint64_t>();
    if (local.n_rows) {
        pack_rowinfo_kernel<<<(unsigned)std::min<uint64_t>((local.n_rows + 255) / 256, 148 * 8), 256, 0, ctx.stream>>>(
            local.d_offsets.as<uint64_t>(), local.d_nums.as<uint32_t>(), local.n_rows, my_info);
        SM_LAUNCHED();
    }
    SM_CUDA(cudaMemsetAsync(all_lens + n_rows, 0, 8, ctx.stream));
    SM_CUDA(cudaEventRecord(c.ev_ready, ctx.stream));       // buffers allocated (stream-ordered) and records packed
    SM_CUDA(cudaStreamWaitEvent(c.stream, c.ev_ready, 0));
    SM_NCCL(g_nccl.GroupStart());
    allgatherv(local.d_hashes.p, out->d_hashes.p, hashes, hash_base, 8, ncclUint64);
    allgatherv(my_info, all_info, rows, row_base, 8, ncclUint64);
    SM_NCCL(g_nccl.GroupEnd());
    SM_CUDA(cudaEventRecord(c.ev_done, c.stream));
    SM_CUDA(cudaStreamWaitEvent(ctx.stream, c.ev_done, 0));
    if (n_rows) {
        unpack_rowinfo_kernel<<<(unsigned)std::min<uint64_t>((n_rows + 255) / 256, 148 * 8), 256, 0, ctx.stream>>>(
            all_info, n_rows, all_lens, out->d_nums.as<uint32_t>());
        SM_LAUNCHED();
    }
    // (scan scratch: join[5], not scan_tmp -- compare_matrix_allgather's table build may be using that on its own stream)
    ctx.join[5].reserve(scan_tmp_bytes(n_rows + 1) + 256);
    scan_exclusive_u64(all_lens, out->d_offsets.as<uint64_t>(), n_rows + 1, ctx.join[5].p, ctx.stream);
    // host mirrors the block logic sizes its work from (collection.cu)
    out->h_offsets.resize(n_rows + 1);
    out->h_nums.resize(n_rows);
    SM_CUDA(cudaMemcpyAsync(out->h_offsets.data(), out->d_offsets.p, (n_rows + 1) * 8, cudaMemcpyDeviceToHost, ctx.stream));
    if (n_rows) SM_CUDA(cudaMemcpyAsync(out->h_nums.data(), out->d_nums.p, n_rows * 4, cudaMemcpyDeviceToHost, ctx.stream));
    ctx.sync();
    if (out->h_offsets[n_rows] != n_hashes) throw_internal("all-gather: row lengths and hash counts disagree");
    out->dirty = false;
    return out.release();
}

SketchCollection *collection_allgather(SketchCollection &local) {
    std::lock_guard<std::mutex> lk(g_comm_mutex);
    return allgather_impl(local, nullptr);
}

// rows of `local` x rows of every rank (rank order): the row block this rank owns of the all-vs-all matrix.
SketchCollection *compare_matrix_allgather(SketchCollection &local, int mode, uint32_t *common, uint32_t *size, double *ratio,
                                           uint64_t ld, bool out_on_device) {
    std::lock_guard<std::mutex> lk(g_comm_mutex);
    Context &ctx = Context::get();
    local.finalize();
    JoinTable jt;
    // The hash table of the join goes over this rank's OWN rows: build it while the other ranks' rows are in flight.
    // (Only when the block will take the probe form of the join: collection.cu decides the same way.)
    const uint64_t n_rp = local.n_hashes;
    const bool will_probe = probe_form_allowed(local) && n_rp < (1ull << 31) && local.n_rows < (1ull << 31);
    // (device outputs, probe form: the gathered rows may still be arriving when the block starts -- see allgather_impl)
    cudaEvent_t cols_ready = nullptr;
    const bool alone = !g_comm.comm || g_comm.world == 1;   // one rank: rows and columns are the same sketches
    // Queued while the headers are on their way and on a stream of its own: neither the host round trip of the headers
    // nor the transfer (whose buffers are allocated in this thread's stream order) waits for it.  Whatever happens below, this
    // thread's stream waits for the build before it goes on (the table lives in the thread's scratch).
    struct JoinBuild {
        cudaStream_t st = nullptr;
        void join() {
            if (st && cudaStreamWaitEvent(st, g_comm.ev_build_done, 0) != cudaSuccess) (void)cudaGetLastError();
            st = nullptr;
        }
        ~JoinBuild() { join(); }
    } join_build;
    auto build_table = [&]() {
        if (!will_probe) return;
        const bool beside = !alone;
        join_table_build(ctx, jt, local.d_hashes.as<uint64_t>(), local.d_offsets.as<uint64_t>(), 0, local.n_rows, n_rp,
                         g_comm.world >= 4, beside ? g_comm.build_stream : nullptr, g_comm.ev_build_go);
        if (beside) {
            SM_CUDA(cudaEventRecord(g_comm.ev_build_done, g_comm.build_stream));
            join_build.st = ctx.stream;
        }
    };
    std::unique_ptr<SketchCollection> all(allgather_impl(local, build_table, (will_probe && out_on_device && !alone) ? &cols_ready : nullptr));
    join_build.join();
    const uint64_t nr = local.n_rows, nc = all->n_rows;
    try {
        local.check_compatible(*all);
        if (nr != 0 && nc != 0 && ld < nc) throw_internal("ld smaller than the block width");
    } catch (...) {
        if (cols_ready) SM_CUDA(cudaStreamWaitEvent(ctx.stream, cols_ready, 0));   // (the gathered buffers are released in stream order)
        throw;
    }
    if (nr == 0 || nc == 0) {
        if (cols_ready) SM_CUDA(cudaStreamWaitEvent(ctx.stream, cols_ready, 0));
        return all.release();
    }
    if (out_on_device) {
        try {
            compare_block_device(local, 0, nr, alone ? local : *all, 0, nc, mode, common, size, ratio, ld, &jt, cols_ready);
        } catch (...) {
            if (cols_ready) SM_CUDA(cudaStreamWaitEvent(ctx.stream, cols_ready, 0));
            throw;
        }
        ctx.sync();
    } else if (alone) {
        compare_matrix(local, 0, nr, local, 0, nc, mode, common, size, ratio, ld, out_on_device);
    } else {
        // host output: row blocks through device scratch, copied back while the next block runs (a block covers
        // part of the rows only, so the table built above does not apply)
        compare_matrix(local, 0, nr, *all, 0, nc, mode, common, size, ratio, ld, out_on_device);
    }
    return all.release();
}

// ---------------------------------------------------------------------------------------------------------
// the partial sketches of one sample, one per rank -> their merge, on every rank (rank order; lib.rs:307-403)
// ---------------------------------------------------------------------------------------------------------
void comm_allmerge(KmerMinHash &mh) {
    std::lock_guard<std::mutex> lk(g_comm_mutex);
    Comm &c = g_comm;
    if (!c.comm || c.world == 1) return;  // a world of one: nothing to combine
    Context &ctx = Context::get();
    size_t n_m = 0, n_a = 0;
    const uint64_t *d_m = mh.device_mins(&n_m);
    const uint64_t *d_a = mh.device_abunds(&n_a);
    const bool track = mh.track_abundance();
    unsigned long long mine[HDR] = {n_m, track ? n_a : 0, track, mh.ksize, mh.seed, mh.max_hash, mh.is_protein, mh.num};
    exchange_headers(mine);
    const int W = c.world;
    std::vector<uint64_t> cm(W), ca(W), bm(W), ba(W);
    uint64_t tm = 0, ta = 0;
    for (int r = 0; r < W; r++) {
        const unsigned long long *h = c.h_hdr + (size_t)r * HDR;
        if (h[3] != mh.ksize) throw SourmashError(ERR_MISMATCH_KSIZES, "different ksizes cannot be compared");
        if ((bool)h[6] != mh.is_protein) throw SourmashError(ERR_MISMATCH_DNAPROT, "DNA/prot minhashes cannot be compared");
        if (h[5] != mh.max_hash) throw SourmashError(ERR_MISMATCH_MAXHASH, "mismatch in max_hash; comparison fail");
        if (h[4] != mh.seed) throw SourmashError(ERR_MISMATCH_SEED, "mismatch in seed; comparison fail");
        cm[r] = h[0]; ca[r] = h[1]; bm[r] = tm; ba[r] = ta;
        tm += h[0]; ta += h[1];
    }
    ctx.misc[6].reserve((tm + 1) * 8);
    ctx.misc[7].reserve((ta + 1) * 8);
    SM_CUDA(cudaEventRecord(c.ev_ready, ctx.stream));
    SM_CUDA(cudaStreamWaitEvent(c.stream, c.ev_ready, 0));
    SM_NCCL(g_nccl.GroupStart());
    allgatherv(d_m, ctx.misc[6].p, cm, bm, 8, ncclUint64);
    allgatherv(d_a, ctx.misc[7].p, ca, ba, 8, ncclUint64);
    SM_NCCL(g_nccl.GroupEnd());
    std::vector<uint64_t> all_m(tm), all_a(ta);
    if (tm) SM_CUDA(cudaMemcpyAsync(all_m.data(), ctx.misc[6].p, tm * 8, cudaMemcpyDeviceToHost, c.stream));
    if (ta) SM_CUDA(cudaMemcpyAsync(all_a.data(), ctx.misc[7].p, ta * 8, cudaMemcpyDeviceToHost, c.stream));
    SM_CUDA(cudaStreamSynchronize(c.stream));
    // acc = sketch of rank 0; acc.merge(sketch of rank 1); ... -- the same fold on every rank
    KmerMinHash acc(mh.num, mh.ksize, mh.is_protein, mh.seed, mh.max_hash, c.h_hdr[2] != 0);
    acc.set_from_host(all_m.data() + bm[0], cm[0], c.h_hdr[2] ? all_a.data() + ba[0] : nullptr, ca[0]);
    for (int r = 1; r < W; r++) {
        const unsigned long long *h = c.h_hdr + (size_t)r * HDR;
        KmerMinHash part(mh.num, mh.ksize, mh.is_protein, mh.seed, mh.max_hash, h[2] != 0);
        part.set_from_host(all_m.data() + bm[r], cm[r], h[2] ? all_a.data() + ba[r] : nullptr, ca[r]);
        acc.merge(part);
    }
    mh.take_state_of(acc);
}

// ---------------------------------------------------------------------------------------------------------
// LinearIndex::find over an index partitioned by rank (rank r holds the rows after those of ranks < r)
// ---------------------------------------------------------------------------------------------------------
uint64_t linear_find_sharded(SketchCollection &index_part, SketchCollection &queries, int mode, double threshold,
                             uint64_t *hit_offsets, uint64_t *hits, uint64_t hits_cap) {
    std::lock_guard<std::mutex> lk(g_comm_mutex);
    Comm &c = g_comm;
    if (!c.comm) return linear_find(index_part, queries, mode, threshold, hit_offsets, hits, hits_cap);  // a world of one
    Context &ctx = Context::get();
    queries.finalize();
    const uint64_t nq = queries.n_rows;
    // local search: hit lists with local row ids
    std::vector<std::vector<uint64_t>> lists = linear_find_lists(index_part, queries, mode, threshold);
    std::vector<uint64_t> loc_off(nq + 1, 0), loc_hits;
    for (uint64_t q = 0; q < nq; q++) {
        loc_hits.insert(loc_hits.end(), lists[q].begin(), lists[q].end());
        loc_off[q + 1] = loc_hits.size();
    }
    const uint64_t n_loc = loc_hits.size();
    unsigned long long mine[HDR] = {index_part.n_rows, n_loc, nq, 0, 0, 0, 0, 0};
    exchange_headers(mine);
    const int W = c.world;
    std::vector<uint64_t> cnt_h(W), cnt_o(W), base_h(W), base_o(W), row_base(W);
    uint64_t th = 0, rows_before = 0;
    for (int r = 0; r < W; r++) {
        const unsigned long long *h = c.h_hdr + (size_t)r * HDR;
        if (h[2] != nq) throw_internal("linear_find_sharded: ranks hold different query batches");
        row_base[r] = rows_before; rows_before += h[0];
        cnt_h[r] = h[1]; base_h[r] = th; th += h[1];
        cnt_o[r] = nq + 1; base_o[r] = (uint64_t)r * (nq + 1);
    }
    // my hits (global ids) and offsets to the device, all-gather, back to the host
    ctx.misc[4].reserve((n_loc + nq + 2) * 8);
    ctx.misc[5].reserve((th + 1) * 8);
    ctx.misc[6].reserve(((uint64_t)W * (nq + 1) + 1) * 8);
    uint64_t *d_my_hits = ctx.misc[4].as<uint64_t>(), *d_my_off = d_my_hits + n_loc;
    if (n_loc) SM_CUDA(cudaMemcpyAsync(d_my_hits, loc_hits.data(), n_loc * 8, cudaMemcpyHostToDevice, ctx.stream));
    SM_CUDA(cudaMemcpyAsync(d_my_off, loc_off.data(), (nq + 1) * 8, cudaMemcpyHostToDevice, ctx.stream));
    if (n_loc && row_base[c.rank]) {
        add_base_kernel<<<(unsigned)std::min<uint64_t>((n_loc + 255) / 256, 148 * 8), 256, 0, ctx.stream>>>(d_my_hits, n_loc, row_base[c.rank]);
        SM_LAUNCHED();
    }
    SM_CUDA(cudaEventRecord(c.ev_ready, ctx.stream));
    SM_CUDA(cudaStreamWaitEvent(c.stream, c.ev_ready, 0));
    SM_NCCL(g_nccl.GroupStart());
    allgatherv(d_my_hits, ctx.misc[5].p, cnt_h, base_h, 8, ncclUint64);
    allgatherv(d_my_off, ctx.misc[6].p, cnt_o, base_o, 8, ncclUint64);
    SM_NCCL(g_nccl.GroupEnd());
    std::vector<uint64_t> all_hits(std::max<uint64_t>(1, th)), all_off((size_t)W * (nq + 1));
    if (th) SM_CUDA(cudaMemcpyAsync(all_hits.data(), ctx.misc[5].p, th * 8, cudaMemcpyDeviceToHost, c.stream));
    SM_CUDA(cudaMemcpyAsync(all_off.data(), ctx.misc[6].p, all_off.size() * 8, cudaMemcpyDeviceToHost, c.stream));
    SM_CUDA(cudaStreamSynchronize(c.stream));
    ctx.sync();
    // per query: the parts' lists in partition order = the insertion order of the whole index (linear.rs:34-44)
    uint64_t total = 0;
    for (uint64_t q = 0; q < nq; q++) {
        if (hit_offsets) hit_offsets[q] = total;
        for (int r = 0; r < W; r++) {
            const uint64_t *off = all_off.data() + (size_t)r * (nq + 1);
            for (uint64_t i = off[q]; i < off[q + 1]; i++) {
                if (hits && total < hits_cap) hits[total] = all_hits[base_h[r] + i];
                total++;
            }
        }
    }
    if (hit_offsets) hit_offsets[nq] = total;
    return total;
}

}  // namespace smb200
