// comm.cu — the one collective on this path: LOLA overlap-count matrices with the database sharded by region set.
//
// Every rank (one process per GPU) holds a gtgpu_igd over its own slice of the database's region sets, computes its
// column block of the [n_sets x n_files] matrix, and the blocks are combined with ONE ncclAllGather over
// NVLink / NVSwitch, enqueued on the compute stream right behind the count kernel (no host synchronisation in
// between); a small kernel then transposes the gathered blocks into the row-major matrix the reference returns.
// Tokenize / count / find shard by query and need no collective at all (SURVEY.md §8e).
//
// NCCL is bound at run time (dlopen of libnccl.so.2) so that single-GPU users never load it and so that a process
// which already carries torch's bundled NCCL reuses that copy.
#include <dlfcn.h>
#include <nccl.h>

#include <algorithm>
#include <cstring>

#include "common.cuh"

#include <functional>

namespace gtgpu {

struct NcclApi {
    void* lib = nullptr;
    ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
    ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
    ncclResult_t (*CommInitAll)(ncclComm_t*, int, const int*) = nullptr;
    ncclResult_t (*AllGather)(const void*, void*, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    const char* (*GetErrorString)(ncclResult_t) = nullptr;
};

static NcclApi* nccl_api() {
    static NcclApi api;
    static bool tried = false;
    if (!tried) {
        tried = true;
        const char* names[] = {"libnccl.so.2", "libnccl.so"};
        for (const char* nm : names) {
            api.lib = dlopen(nm, RTLD_NOW | RTLD_GLOBAL);
            if (api.lib) break;
        }
        if (api.lib) {
            api.GetUniqueId = (decltype(api.GetUniqueId))dlsym(api.lib, "ncclGetUniqueId");
            api.CommInitRank = (decltype(api.CommInitRank))dlsym(api.lib, "ncclCommInitRank");
            api.CommInitAll = (decltype(api.CommInitAll))dlsym(api.lib, "ncclCommInitAll");
            api.AllGather = (decltype(api.AllGather))dlsym(api.lib, "ncclAllGather");
            api.CommDestroy = (decltype(api.CommDestroy))dlsym(api.lib, "ncclCommDestroy");
            api.GetErrorString = (decltype(api.GetErrorString))dlsym(api.lib, "ncclGetErrorString");
            if (!api.GetUniqueId || !api.CommInitRank || !api.AllGather || !api.CommDestroy) api.lib = nullptr;
        }
    }
    return api.lib ? &api : nullptr;
}

struct Comm {
    ncclComm_t comm = nullptr;
    int world = 1, rank = 0;
};

// gathered[r][s][j] (j < cols_per_rank) -> out[s][r * cols_per_rank + j] for columns that exist
__global__ void untranspose_blocks_kernel(uint32_t world, uint64_t n_sets, uint64_t cols_per_rank, uint64_t n_files,
                                          const uint64_t* __restrict__ gathered, uint64_t* __restrict__ out) {
    const uint64_t total = n_sets * n_files;
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t k = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; k < total; k += stride) {
        const uint64_t s = k / n_files, f = k % n_files;
        const uint64_t r = f / cols_per_rank, j = f % cols_per_rank;
        out[k] = gathered[(r * n_sets + s) * cols_per_rank + j];
    }
}

}  // namespace gtgpu

using namespace gtgpu;

#define GT_NCCL(api, expr)                                                                                           \
    do {                                                                                                             \
        ncclResult_t _r = (expr);                                                                                    \
        if (_r != ncclSuccess)                                                                                       \
            return fail(GTGPU_ERR_NCCL, std::string(#expr) + ": " + ((api)->GetErrorString ? (api)->GetErrorString(_r) : "?")); \
    } while (0)

extern "C" int32_t gtgpu_comm_unique_id(uint8_t out_id[128]) try {
    if (!out_id) return fail(GTGPU_ERR_INVALID, "comm_unique_id: null argument");
    NcclApi* api = nccl_api();
    if (!api) return fail(GTGPU_ERR_NCCL, "libnccl.so.2 could not be loaded");
    ncclUniqueId id;
    GT_NCCL(api, api->GetUniqueId(&id));
    static_assert(sizeof(ncclUniqueId) == 128, "ncclUniqueId is 128 bytes");
    memcpy(out_id, &id, 128);
    return GTGPU_OK;
} GT_CATCH

extern "C" int32_t gtgpu_comm_init(gtgpu_ctx* ctx, int32_t world, int32_t rank, const uint8_t id_bytes[128]) try {
    if (!ctx || !id_bytes || world < 1 || rank < 0 || rank >= world) return fail(GTGPU_ERR_INVALID, "comm_init: bad argument");
    NcclApi* api = nccl_api();
    if (!api) return fail(GTGPU_ERR_NCCL, "libnccl.so.2 could not be loaded");
    std::lock_guard<std::mutex> lk(ctx->mu);
    GT_CUDA(cudaSetDevice(ctx->device));
    if (ctx->comm) return fail(GTGPU_ERR_INVALID, "comm_init: communicator already initialised");
    if (ctx->peers.size() > 1) return fail(GTGPU_ERR_INVALID, "comm_init: a multi-device context creates its own communicators");
    ncclUniqueId id;
    memcpy(&id, id_bytes, 128);
    Comm* c = new Comm();
    c->world = world;
    c->rank = rank;
    ncclResult_t r = api->CommInitRank(&c->comm, world, id, rank);
    if (r != ncclSuccess) {
        delete c;
        return fail(GTGPU_ERR_NCCL, std::string("ncclCommInitRank: ") + (api->GetErrorString ? api->GetErrorString(r) : "?"));
    }
    ctx->comm = c;
    return GTGPU_OK;
} GT_CATCH

extern "C" int32_t gtgpu_comm_free(gtgpu_ctx* ctx) try {
    if (!ctx || !ctx->comm) return GTGPU_OK;
    NcclApi* api = nccl_api();
    Comm* c = (Comm*)ctx->comm;
    if (api && c->comm) api->CommDestroy(c->comm);
    delete c;
    ctx->comm = nullptr;
    return GTGPU_OK;
} GT_CATCH

// In-process communicators for a multi-device group: one ncclComm per peer ctx (ncclCommInitAll), created on first use.
int32_t gtgpu::group_comm_ensure(gtgpu_ctx* g) {
    if (g->peers.size() < 2) return GTGPU_OK;
    if (g->group_comm_tried) return g->peers[0]->comm ? GTGPU_OK : fail(GTGPU_ERR_NCCL, "group communicators could not be created");
    g->group_comm_tried = true;
    NcclApi* api = nccl_api();
    if (!api || !api->CommInitAll) return fail(GTGPU_ERR_NCCL, "libnccl.so.2 could not be loaded");
    const int n = (int)g->peers.size();
    std::vector<ncclComm_t> comms(n);
    std::vector<int> devs(n);
    for (int r = 0; r < n; ++r) devs[r] = g->peers[r]->device;
    GT_NCCL(api, api->CommInitAll(comms.data(), n, devs.data()));
    for (int r = 0; r < n; ++r) {
        Comm* c = new Comm();
        c->comm = comms[r];
        c->world = n;
        c->rank = r;
        g->peers[r]->comm = c;
    }
    return GTGPU_OK;
}

// Database sharded by region set: rank r owns global files [r * cols, min((r+1) * cols, n_files_global)),
// cols = ceil(n_files_global / world); `igd` was built over exactly those files (possibly none).  chr / start / end may be
// host memory or device memory of any device (cudaMemcpyDefault); set_offsets is host memory.  `out` may be null (a
// peer of an in-process group: only the first device returns the matrix); before_collective, when given, runs right
// before the all-gather is queued (groups use it as a barrier so that no thread is still allocating device memory while
// another one's collective kernel already waits for it).
int32_t gtgpu::igd_count_sharded_impl(gtgpu_ctx* ctx, gtgpu_igd* igd, int32_t binary, uint64_t n_files_global, uint64_t n_sets,
                                      const uint64_t* set_offsets, const uint32_t* chr, const uint32_t* start, const uint32_t* end,
                                      int32_t min_overlap, uint64_t* out, const std::function<bool(bool)>* before_collective) {
    // Everything in front of the collective runs inside `prepare`; a group then meets at before_collective(ok), which
    // tells every device whether ALL of them got this far — a device that failed must not leave the others waiting
    // inside an all-gather it will never join.
    std::unique_lock<std::mutex> lk;
    Comm* c = nullptr;
    int world = 1, rank = 0;
    uint64_t cols = 0, n = 0;
    uint64_t *d_local = nullptr, *d_gather = nullptr, *d_full = nullptr;
    cudaStream_t st = nullptr;
    NcclApi* api = nullptr;
    auto prepare = [&]() -> int32_t {
        if (!ctx || !igd || !set_offsets) return fail(GTGPU_ERR_INVALID, "igd_count_sharded: null argument");
        if (igd->ctx != ctx) return fail(GTGPU_ERR_INVALID, "igd_count_sharded: the igd was built on another context");
        for (uint64_t s = 0; s < n_sets; ++s)
            if (set_offsets[s] > set_offsets[s + 1]) return fail(GTGPU_ERR_INVALID, "igd_count_sharded: set_offsets not monotone");
        lk = std::unique_lock<std::mutex>(ctx->mu);  // held for the whole call: no other call can grow (= move) the scratch
        c = (Comm*)ctx->comm;
        world = c ? c->world : 1;
        rank = c ? c->rank : 0;
        cols = (n_files_global + world - 1) / world;
        const uint64_t lo = std::min<uint64_t>((uint64_t)rank * cols, n_files_global);
        const uint64_t hi = std::min<uint64_t>(lo + cols, n_files_global);
        if (igd->n_files != hi - lo) return fail(GTGPU_ERR_INVALID, "igd_count_sharded: this rank's igd does not hold its slice of the sets");
        n = set_offsets[n_sets];
        if (n && (!chr || !start || !end)) return fail(GTGPU_ERR_INVALID, "igd_count_sharded: null query arrays");
        if (min_overlap < 1) return fail(GTGPU_ERR_UNSUPPORTED, "igd count: min_overlap < 1 depends on the reference's tile layout and is not supported");
        api = world > 1 ? nccl_api() : nullptr;
        if (world > 1 && !api) return fail(GTGPU_ERR_NCCL, "libnccl.so.2 could not be loaded");
        GT_CUDA(cudaSetDevice(ctx->device));
        st = ctx->stream;
        uint32_t *d_chr, *d_start, *d_end, *d_set;
        uint64_t *d_so, *d_tmp = nullptr;
        const uint64_t local = hi - lo;
        GT_TRY(ctx->scratch_get(SC_CHR, n * 4, (void**)&d_chr));
        GT_TRY(ctx->scratch_get(SC_START, n * 4, (void**)&d_start));
        GT_TRY(ctx->scratch_get(SC_END, n * 4, (void**)&d_end));
        GT_TRY(ctx->scratch_get(SC_SET_ID, n * 4, (void**)&d_set));
        GT_TRY(ctx->scratch_get(SC_FILE_OFFS, (n_sets + 1) * 8, (void**)&d_so));
        GT_TRY(ctx->scratch_get(SC_MATRIX, n_sets * cols * 8 + 8, (void**)&d_local));
        GT_TRY(ctx->scratch_get(SC_IN3_CHR, (uint64_t)world * n_sets * cols * 8 + 8, (void**)&d_gather));
        GT_TRY(ctx->scratch_get(SC_IN3_START, n_sets * n_files_global * 8 + 8, (void**)&d_full));
        if (local != cols) GT_TRY(ctx->scratch_get(SC_IN3_END, n_sets * local * 8 + 8, (void**)&d_tmp));
        if (n) {  // host arrays, or (a group counting parsed BED files) the first device's columns
            GT_CUDA(cudaMemcpyAsync(d_chr, chr, n * 4, cudaMemcpyDefault, st));
            GT_CUDA(cudaMemcpyAsync(d_start, start, n * 4, cudaMemcpyDefault, st));
            GT_CUDA(cudaMemcpyAsync(d_end, end, n * 4, cudaMemcpyDefault, st));
        }
        GT_CUDA(cudaMemcpyAsync(d_so, set_offsets, (n_sets + 1) * 8, cudaMemcpyHostToDevice, st));
        GT_CUDA(cudaMemsetAsync(d_local, 0, n_sets * cols * 8 + 8, st));
        // The local block is computed with row stride = the igd's own file count; make that equal to `cols` by padding:
        // ranks whose slice is shorter than `cols` (the last one) count into a [n_sets x local] matrix first.
        uint64_t* d_cnt = d_local;
        if (local != cols) {
            GT_CUDA(cudaMemsetAsync(d_tmp, 0, n_sets * local * 8 + 8, st));
            d_cnt = d_tmp;
        }
        if (n && n_sets) {
            GT_TRY(launch_fill_set_ids(ctx, n_sets, d_so, d_set));
            if (local) GT_TRY(igd_count_dev_locked(igd, binary != 0, n, d_set, d_chr, d_start, d_end, min_overlap, d_cnt));
        }
        if (local != cols && local)
            GT_CUDA(cudaMemcpy2DAsync(d_local, cols * 8, d_tmp, local * 8, local * 8, n_sets, cudaMemcpyDeviceToDevice, st));
        return GTGPU_OK;
    };
    int32_t status;
    try {
        status = prepare();
    } catch (...) {
        status = translate_exception();
    }
    if (before_collective) {
        std::string msg = status != GTGPU_OK ? std::string(gtgpu_last_error()) : std::string();
        const bool all_ok = (*before_collective)(status == GTGPU_OK);
        if (status != GTGPU_OK) return fail(status, msg);
        if (!all_ok) return fail(GTGPU_ERR_NCCL, "igd count: another device of the group failed before the collective");
    } else if (status != GTGPU_OK) {
        return status;
    }
    const uint64_t* d_src = d_local;
    if (world > 1) {
        GT_NCCL(api, api->AllGather(d_local, d_gather, n_sets * cols, ncclUint64, c->comm, st));
        d_src = d_gather;
    }
    const uint64_t cells = n_sets * n_files_global;
    if (cells && out) {
        int grid = (int)std::min<uint64_t>((cells + 255) / 256, (uint64_t)ctx->sm_count * 16);
        untranspose_blocks_kernel<<<grid, 256, 0, st>>>((uint32_t)world, n_sets, cols, n_files_global, d_src, d_full);
        ctx->launches++;
        GT_CUDA(cudaMemcpyAsync(out, d_full, cells * 8, cudaMemcpyDeviceToHost, st));
    }
    GT_CUDA(cudaStreamSynchronize(st));
    return GTGPU_OK;
}

extern "C" int32_t gtgpu_igd_count_sharded(gtgpu_ctx* ctx, gtgpu_igd* igd, int32_t binary, uint64_t n_files_global,
                                           uint64_t n_sets, const uint64_t* set_offsets, const uint32_t* chr,
                                           const uint32_t* start, const uint32_t* end, int32_t min_overlap, uint64_t* out) try {
    if (!out) return fail(GTGPU_ERR_INVALID, "igd_count_sharded: null argument");
    if (ctx && ctx->peers.size() > 1) return fail(GTGPU_ERR_INVALID, "igd_count_sharded: a multi-device context shards inside gtgpu_igd_count_*");
    return igd_count_sharded_impl(ctx, igd, binary, n_files_global, n_sets, set_offsets, chr, start, end, min_overlap, out, nullptr);
} GT_CATCH
