// api.cu — extern "C" entry points of include/gtars_gpu.h: context, memory, and the host-buffer wrappers
// (H2D → kernels → D2H) around the device-resident launches in kernels.cu.
#include <algorithm>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <memory>
#include <thread>
#include <vector>

#include "common.cuh"

namespace gtgpu {

static thread_local std::string g_last_error;

void set_error(const std::string& msg) { g_last_error = msg; }
int32_t fail(int32_t code, const std::string& msg) {
    g_last_error = msg;
    return code;
}

// Called from a catch (...) handler of an entry point: classify the in-flight exception without letting it escape.
int32_t translate_exception() noexcept {
    try {
        try {
            throw;
        } catch (const std::bad_alloc&) {
            g_last_error = "out of host memory (std::bad_alloc)";
            return GTGPU_ERR_NOMEM;
        } catch (const std::exception& e) {
            g_last_error = std::string("unexpected C++ exception: ") + e.what();
            return GTGPU_ERR_INVALID;
        } catch (...) {
            g_last_error = "unexpected non-standard exception";
            return GTGPU_ERR_INVALID;
        }
    } catch (...) {  // building the message itself failed
        return GTGPU_ERR_NOMEM;
    }
}

// fn(r) for every device r of a group, one host thread per device (r = 0 on the caller's); the first failure wins and
// its message becomes the caller's last_error (error text is thread-local).
int32_t for_each_device(size_t n_devices, const std::function<int32_t(size_t)>& fn) {
    std::vector<int32_t> st(n_devices, GTGPU_OK);
    std::vector<std::string> msg(n_devices);
    auto run = [&](size_t r) {
        try {
            st[r] = fn(r);
        } catch (...) {
            st[r] = translate_exception();
        }
        if (st[r] != GTGPU_OK) msg[r] = g_last_error;
    };
    std::vector<std::thread> th;
    for (size_t r = 1; r < n_devices; ++r) th.emplace_back(run, r);
    run(0);
    for (auto& t : th) t.join();
    for (size_t r = 0; r < n_devices; ++r)
        if (st[r] != GTGPU_OK) return fail(st[r], msg[r]);
    return GTGPU_OK;
}

// contiguous block r of n items over `world` shards: sizes differ by at most one, earlier shards get the larger blocks
void block_range(uint64_t n, uint64_t world, uint64_t r, uint64_t* lo, uint64_t* hi) {
    const uint64_t base = n / world, extra = n % world;
    *lo = r * base + std::min(r, extra);
    *hi = *lo + base + (r < extra ? 1 : 0);
}

}  // namespace gtgpu

using namespace gtgpu;

// ---- ctx members ---------------------------------------------------------------------------------------------------
int32_t gtgpu_ctx::scratch_get(int role, size_t bytes, void** out) {
    if (scratch.size() < (size_t)SC_N_ROLES) scratch.resize(SC_N_ROLES);
    DevBuffer& b = scratch[role];
    bytes = std::max<size_t>(bytes, 256);
    if (b.cap < bytes) {
        if (b.ptr) cudaFree(b.ptr);
        b.ptr = nullptr;
        b.cap = 0;
        size_t want = bytes + bytes / 16;  // a little slack so slowly growing batches do not realloc every call
        cudaError_t e = cudaMalloc(&b.ptr, want);
        if (e != cudaSuccess) {
            want = bytes;
            e = cudaMalloc(&b.ptr, want);
        }
        if (e != cudaSuccess)
            return fail(GTGPU_ERR_NOMEM, "cudaMalloc(" + std::to_string(bytes) + " B): " + cudaGetErrorString(e));
        b.cap = want;
    }
    *out = b.ptr;
    return GTGPU_OK;
}

int32_t gtgpu_ctx::pinned_get(size_t bytes, PinnedBlock* out) {
    bytes = std::max<size_t>(bytes, 64);
    std::lock_guard<std::mutex> lk(pinned_mu);
    int best = -1;
    for (size_t i = 0; i < pinned_free.size(); ++i)
        if (pinned_free[i].cap >= bytes && (best < 0 || pinned_free[i].cap < pinned_free[best].cap)) best = (int)i;
    if (best >= 0) {
        *out = pinned_free[best];
        pinned_free.erase(pinned_free.begin() + best);
        return GTGPU_OK;
    }
    PinnedBlock b;
    cudaError_t e = cudaHostAlloc(&b.ptr, bytes, cudaHostAllocDefault);
    if (e != cudaSuccess) {
        // free the cache and retry once
        for (auto& f : pinned_free) cudaFreeHost(f.ptr);
        pinned_free.clear();
        e = cudaHostAlloc(&b.ptr, bytes, cudaHostAllocDefault);
    }
    if (e != cudaSuccess)
        return fail(GTGPU_ERR_NOMEM, "cudaHostAlloc(" + std::to_string(bytes) + " B): " + cudaGetErrorString(e));
    b.cap = bytes;
    *out = b;
    return GTGPU_OK;
}

void gtgpu_ctx::pinned_put(PinnedBlock b) {
    if (!b.ptr) return;
    std::lock_guard<std::mutex> lk(pinned_mu);
    pinned_free.push_back(b);
    // keep at most 8 blocks; drop the smallest first
    while (pinned_free.size() > 8) {
        size_t k = 0;
        for (size_t i = 1; i < pinned_free.size(); ++i)
            if (pinned_free[i].cap < pinned_free[k].cap) k = i;
        cudaFreeHost(pinned_free[k].ptr);
        pinned_free.erase(pinned_free.begin() + k);
    }
}

int32_t gtgpu::buf_new(gtgpu_ctx* ctx, uint64_t len, uint32_t elem_size, BufPtr* out) {
    BufPtr buf(new (std::nothrow) gtgpu_buf());
    if (!buf) return fail(GTGPU_ERR_NOMEM, "out of host memory (result buffer)");
    buf->ctx = ctx;
    buf->len = len;
    buf->elem_size = elem_size;
    GT_TRY(ctx->pinned_get(len * elem_size, &buf->block));
    *out = std::move(buf);
    return GTGPU_OK;
}

int32_t gtgpu::buf_from_device(gtgpu_ctx* ctx, const void* d_src, uint64_t len, uint32_t elem_size, cudaStream_t st, BufPtr* out) {
    BufPtr buf;
    GT_TRY(buf_new(ctx, len, elem_size, &buf));
    const cudaError_t e = len ? cudaMemcpyAsync(buf->block.ptr, d_src, len * elem_size, cudaMemcpyDeviceToHost, st) : cudaSuccess;
    if (e != cudaSuccess) return fail(GTGPU_ERR_CUDA, cudaGetErrorString(e));
    *out = std::move(buf);
    return GTGPU_OK;
}

void gtgpu_ctx::time_begin() {
    if (!timing || ev_used >= 256) return;
    if (ev_begin.size() <= ev_used) {
        cudaEvent_t a, b;
        cudaEventCreate(&a);
        cudaEventCreate(&b);
        ev_begin.push_back(a);
        ev_end.push_back(b);
    }
    cudaEventRecord(ev_begin[ev_used], stream);
}

void gtgpu_ctx::time_end() {
    if (!timing || ev_used >= 256) return;
    cudaEventRecord(ev_end[ev_used], stream);
    ev_used++;
}

extern "C" {

int32_t gtgpu_timing_enable(gtgpu_ctx* ctx, int32_t on) try {
    if (!ctx) return fail(GTGPU_ERR_INVALID, "timing_enable: null ctx");
    std::lock_guard<std::mutex> lk(ctx->mu);
    ctx->timing = on != 0;
    ctx->ev_used = 0;
    return GTGPU_OK;
} GT_CATCH

int32_t gtgpu_timing_read(gtgpu_ctx* ctx, float* out_ms, uint32_t cap, uint32_t* out_n) try {
    if (!ctx || !out_n || (cap && !out_ms)) return fail(GTGPU_ERR_INVALID, "timing_read: null argument");
    std::lock_guard<std::mutex> lk(ctx->mu);
    GT_CUDA(cudaSetDevice(ctx->device));
    GT_CUDA(cudaStreamSynchronize(ctx->stream));
    for (uint32_t i = 0; i < ctx->ev_used && i < cap; ++i)
        GT_CUDA(cudaEventElapsedTime(out_ms + i, ctx->ev_begin[i], ctx->ev_end[i]));
    *out_n = ctx->ev_used;
    ctx->ev_used = 0;
    return GTGPU_OK;
} GT_CATCH

const char* gtgpu_last_error(void) { return g_last_error.c_str(); }
const char* gtgpu_version(void) { return "gtars-b200 0.1 (sm_100a)"; }

int32_t gtgpu_device_count(int32_t* out_n) try {
    if (!out_n) return fail(GTGPU_ERR_INVALID, "device_count: null argument");
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess) {
        *out_n = 0;
        return fail(GTGPU_ERR_CUDA, std::string("cudaGetDeviceCount: ") + cudaGetErrorString(e));
    }
    *out_n = n;
    return GTGPU_OK;
} GT_CATCH

static void ctx_destroy(gtgpu_ctx* ctx) {
    cudaSetDevice(ctx->device);
    gtgpu_comm_free(ctx);
    if (ctx->stream) cudaStreamSynchronize(ctx->stream);
    for (auto& b : ctx->scratch)
        if (b.ptr) cudaFree(b.ptr);
    for (auto& b : ctx->pinned_free) cudaFreeHost(b.ptr);
    for (auto e : ctx->ev_begin) cudaEventDestroy(e);
    for (auto e : ctx->ev_end) cudaEventDestroy(e);
    if (ctx->h_scalars) cudaFreeHost(ctx->h_scalars);
    if (ctx->own_stream && ctx->stream) cudaStreamDestroy(ctx->stream);
    if (ctx->copy_in) cudaStreamDestroy(ctx->copy_in);
    if (ctx->copy_out) cudaStreamDestroy(ctx->copy_out);
    delete ctx;
}

static int32_t ctx_create(int32_t device, void* stream_or_null, gtgpu_ctx** out_ctx) {
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0)
        return fail(GTGPU_ERR_CUDA, std::string("no usable CUDA device (there is no CPU fallback): ") +
                                        (e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0"));
    if (device < 0 || device >= n) return fail(GTGPU_ERR_INVALID, "init: device index out of range");
    GT_CUDA(cudaSetDevice(device));
    cudaDeviceProp prop;
    GT_CUDA(cudaGetDeviceProperties(&prop, device));
    if (prop.major < 10)
        return fail(GTGPU_ERR_UNSUPPORTED, std::string("device is sm_") + std::to_string(prop.major * 10 + prop.minor) +
                                               "; this library is built for sm_100a only");
    gtgpu_ctx* ctx = new gtgpu_ctx();
    ctx->device = device;
    ctx->sm_count = prop.multiProcessorCount;
    cudaError_t ce = cudaSuccess;
    if (stream_or_null) {
        ctx->stream = (cudaStream_t)stream_or_null;
    } else {
        ce = cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking);
        ctx->own_stream = ce == cudaSuccess;
    }
    if (ce == cudaSuccess) ce = cudaStreamCreateWithFlags(&ctx->copy_in, cudaStreamNonBlocking);
    if (ce == cudaSuccess) ce = cudaStreamCreateWithFlags(&ctx->copy_out, cudaStreamNonBlocking);
    if (ce == cudaSuccess) ce = cudaHostAlloc((void**)&ctx->h_scalars, 64 * sizeof(uint64_t), cudaHostAllocDefault);
    if (ce != cudaSuccess) {
        ctx_destroy(ctx);  // nothing of a half-built ctx is leaked
        return fail(GTGPU_ERR_CUDA, std::string("init: ") + cudaGetErrorString(ce));
    }
    *out_ctx = ctx;
    return GTGPU_OK;
}

int32_t gtgpu_init(int32_t device, void* stream_or_null, gtgpu_ctx** out_ctx) try {
    if (!out_ctx) return fail(GTGPU_ERR_INVALID, "init: null argument");
    return ctx_create(device, stream_or_null, out_ctx);
} GT_CATCH

int32_t gtgpu_init_multi(int32_t n_devices, const int32_t* device_ids, gtgpu_ctx** out_ctx) try {
    if (!out_ctx || n_devices < 1) return fail(GTGPU_ERR_INVALID, "init_multi: bad argument");
    for (int32_t i = 0; i < n_devices; ++i)
        for (int32_t j = 0; j < i; ++j)
            if (device_ids && device_ids[i] == device_ids[j]) return fail(GTGPU_ERR_INVALID, "init_multi: a device is listed twice");
    std::vector<gtgpu_ctx*> peers;
    for (int32_t i = 0; i < n_devices; ++i) {
        gtgpu_ctx* c = nullptr;
        const int32_t s = ctx_create(device_ids ? device_ids[i] : i, nullptr, &c);
        if (s != GTGPU_OK) {
            for (gtgpu_ctx* p : peers) ctx_destroy(p);
            return s;
        }
        peers.push_back(c);
    }
    if (n_devices > 1) peers[0]->peers = peers;
    *out_ctx = peers[0];
    return GTGPU_OK;
} GT_CATCH

int32_t gtgpu_ctx_devices(const gtgpu_ctx* ctx, int32_t* out_n, int32_t* out_ids, int32_t cap) try {
    if (!ctx || !out_n) return fail(GTGPU_ERR_INVALID, "ctx_devices: null argument");
    const int32_t n = ctx->peers.empty() ? 1 : (int32_t)ctx->peers.size();
    *out_n = n;
    for (int32_t i = 0; out_ids && i < n && i < cap; ++i) out_ids[i] = ctx->peers.empty() ? ctx->device : ctx->peers[i]->device;
    return GTGPU_OK;
} GT_CATCH

int32_t gtgpu_shutdown(gtgpu_ctx* ctx) try {
    if (!ctx) return GTGPU_OK;
    const std::vector<gtgpu_ctx*> peers = ctx->peers;  // copy: ctx dies below
    for (size_t i = 1; i < peers.size(); ++i) ctx_destroy(peers[i]);
    ctx_destroy(ctx);
    return GTGPU_OK;
} GT_CATCH

int32_t gtgpu_synchronize(gtgpu_ctx* ctx) try {
    if (!ctx) return fail(GTGPU_ERR_INVALID, "synchronize: null ctx");
    for (size_t i = 1; i < ctx->peers.size(); ++i) {
        GT_CUDA(cudaSetDevice(ctx->peers[i]->device));
        GT_CUDA(cudaStreamSynchronize(ctx->peers[i]->stream));
    }
    GT_CUDA(cudaSetDevice(ctx->device));
    GT_CUDA(cudaStreamSynchronize(ctx->stream));
    return GTGPU_OK;
} GT_CATCH

int32_t gtgpu_launch_count(gtgpu_ctx* ctx, uint64_t* out_n) try {
    if (!ctx || !out_n) return fail(GTGPU_ERR_INVALID, "launch_count: null argument");
    *out_n = ctx->launches;
    for (size_t i = 1; i < ctx->peers.size(); ++i) *out_n += ctx->peers[i]->launches;
    return GTGPU_OK;
} GT_CATCH

int32_t gtgpu_host_alloc(uint64_t bytes, void** out_ptr) try {
    if (!out_ptr) return fail(GTGPU_ERR_INVALID, "host_alloc: null argument");
    cudaError_t e = cudaHostAlloc(out_ptr, std::max<uint64_t>(bytes, 64), cudaHostAllocDefault);
    if (e != cudaSuccess) return fail(GTGPU_ERR_NOMEM, std::string("cudaHostAlloc: ") + cudaGetErrorString(e));
    return GTGPU_OK;
} GT_CATCH

int32_t gtgpu_host_free(void* ptr) try {
    if (ptr) GT_CUDA(cudaFreeHost(ptr));
    return GTGPU_OK;
} GT_CATCH

const void* gtgpu_buf_data(const gtgpu_buf* buf) { return buf ? buf->block.ptr : nullptr; }
uint64_t gtgpu_buf_len(const gtgpu_buf* buf) { return buf ? buf->len : 0; }
int32_t gtgpu_buf_free(gtgpu_buf* buf) try {
    if (!buf) return GTGPU_OK;
    buf->ctx->pinned_put(buf->block);
    delete buf;
    return GTGPU_OK;
} GT_CATCH

}  // extern "C"

// ---- host-buffer wrappers ------------------------------------------------------------------------------------------
namespace {

struct DevQueries {
    uint32_t *chr = nullptr, *start = nullptr, *end = nullptr;
};

int32_t upload_queries(gtgpu_ctx* ctx, uint64_t n, const uint32_t* chr, const uint32_t* start, const uint32_t* end,
                       DevQueries* q) {
    GT_TRY(ctx->scratch_get(SC_CHR, n * 4, (void**)&q->chr));
    GT_TRY(ctx->scratch_get(SC_START, n * 4, (void**)&q->start));
    GT_TRY(ctx->scratch_get(SC_END, n * 4, (void**)&q->end));
    if (n) {
        GT_CUDA(cudaMemcpyAsync(q->chr, chr, n * 4, cudaMemcpyHostToDevice, ctx->stream));
        GT_CUDA(cudaMemcpyAsync(q->start, start, n * 4, cudaMemcpyHostToDevice, ctx->stream));
        GT_CUDA(cudaMemcpyAsync(q->end, end, n * 4, cudaMemcpyHostToDevice, ctx->stream));
    }
    return GTGPU_OK;
}

int32_t count_host(gtgpu_index* ix, uint64_t n, const uint32_t* chr, const uint32_t* start, const uint32_t* end,
                   int32_t min_overlap, int mode, void* out, size_t elem) {
    if (!ix || (n && (!chr || !start || !end || !out))) return fail(GTGPU_ERR_INVALID, "count: null argument");
    if (mode == COUNT_BITS_RAW_U64 && ix->kind != GTGPU_KIND_BITS)
        return fail(GTGPU_ERR_INVALID, "bits_count: index is not GTGPU_KIND_BITS");
    gtgpu_ctx* ctx = ix->ctx;
    std::lock_guard<std::mutex> lk(ctx->mu);
    GT_CUDA(cudaSetDevice(ctx->device));
    if (n == 0) return GTGPU_OK;
    DevQueries q;
    GT_TRY(upload_queries(ctx, n, chr, start, end, &q));
    void* d_out = nullptr;
    GT_TRY(ctx->scratch_get(SC_COUNTS, n * elem, &d_out));
    GT_TRY(launch_count(ix, n, q.chr, q.start, q.end, min_overlap, mode, d_out));
    GT_CUDA(cudaMemcpyAsync(out, d_out, n * elem, cudaMemcpyDeviceToHost, ctx->stream));
    GT_CUDA(cudaStreamSynchronize(ctx->stream));
    return GTGPU_OK;
}

// Shared body of gtgpu_find (per-query offsets, no files) and gtgpu_tokenize_files (per-file offsets + [unk]).
int32_t find_host(gtgpu_index* ix, uint64_t n, const uint32_t* chr, const uint32_t* start, const uint32_t* end,
                  int32_t min_overlap, uint64_t* out_offsets, bool files, uint64_t n_files,
                  const uint64_t* file_offsets, uint32_t unk_id, uint64_t* out_file_tok, BufPtr* out_ids) {
    gtgpu_ctx* ctx = ix->ctx;
    std::lock_guard<std::mutex> lk(ctx->mu);
    GT_CUDA(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;

    DevQueries q;
    GT_TRY(upload_queries(ctx, n, chr, start, end, &q));
    uint64_t *d_file_offsets = nullptr, *d_raw_tok = nullptr, *d_out_tok = nullptr, *d_offsets = nullptr;
    if (files) {
        GT_TRY(ctx->scratch_get(SC_FILE_OFFS, (n_files + 1) * 8, (void**)&d_file_offsets));
        GT_TRY(ctx->scratch_get(SC_FILE_TOK, (n_files + 1) * 8, (void**)&d_raw_tok));
        GT_TRY(ctx->scratch_get(SC_FILE_TOK2, (n_files + 1) * 8, (void**)&d_out_tok));
        GT_CUDA(cudaMemcpyAsync(d_file_offsets, file_offsets, (n_files + 1) * 8, cudaMemcpyHostToDevice, st));
    } else {
        GT_TRY(ctx->scratch_get(SC_OUT_OFFS, (n + 1) * 8, (void**)&d_offsets));
    }
    void* d_ws = nullptr;
    GT_TRY(ctx->scratch_get(SC_TILE_STATUS, fused_workspace_bytes(n), &d_ws));
    uint64_t* d_misc = nullptr;  // [0] total, [1] n_empty, [2] err flag (u32)
    GT_TRY(ctx->scratch_get(SC_MISC, 64, (void**)&d_misc));

    uint64_t cap = n + n / 4 + 1024;
    uint64_t total = 0, n_empty = 0;
    uint32_t* d_ids = nullptr;
    for (int attempt = 0; attempt < 2; ++attempt) {
        GT_TRY(ctx->scratch_get(SC_OUT_IDS, cap * 4, (void**)&d_ids));
        GT_CUDA(cudaMemsetAsync(d_misc, 0, 64, st));
        GT_TRY(launch_fused_find(ix, n, n_files, d_file_offsets, q.chr, q.start, q.end, min_overlap, d_ids, cap,
                                 d_offsets, d_raw_tok, d_ws, nullptr, d_misc, (uint32_t*)(d_misc + 2)));
        if (files) GT_TRY(launch_unk_offsets(ctx, n_files, d_raw_tok, d_out_tok, d_misc + 1));
        GT_CUDA(cudaMemcpyAsync(ctx->h_scalars, d_misc, 24, cudaMemcpyDeviceToHost, st));
        GT_CUDA(cudaStreamSynchronize(st));
        total = ctx->h_scalars[0];
        n_empty = ctx->h_scalars[1];
        if ((uint32_t)ctx->h_scalars[2] != 0)
            return fail(GTGPU_ERR_UNSUPPORTED, "find: more than 2^32 hits inside one 1024-query tile");
        if (total <= cap) break;
        if (attempt == 1) return fail(GTGPU_ERR_CAPACITY, "find: output capacity exceeded twice");
        cap = total;  // exact re-run
    }

    const uint32_t* d_final = d_ids;
    uint64_t final_total = total;
    if (files && n_empty > 0) {
        uint32_t* d_ids2 = nullptr;
        final_total = total + n_empty;
        GT_TRY(ctx->scratch_get(SC_OUT_IDS2, final_total * 4, (void**)&d_ids2));
        GT_TRY(launch_unk_expand(ctx, n_files, d_raw_tok, d_out_tok, d_ids, unk_id, d_ids2));
        d_final = d_ids2;
    }

    BufPtr buf;
    const int32_t s = buf_from_device(ctx, d_final, final_total, 4, st, &buf);
    if (s == GTGPU_ERR_CUDA) return fail(s, std::string("find: D2H: ") + gtgpu_last_error());
    GT_TRY(s);
    cudaError_t e = cudaSuccess;
    if (files) e = cudaMemcpyAsync(out_file_tok, d_out_tok, (n_files + 1) * 8, cudaMemcpyDeviceToHost, st);
    else e = cudaMemcpyAsync(out_offsets, d_offsets, (n + 1) * 8, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) {
        cudaStreamSynchronize(st);  // the ids' copy may still run
        return fail(GTGPU_ERR_CUDA, std::string("find: D2H: ") + cudaGetErrorString(e));
    }
    *out_ids = std::move(buf);
    return GTGPU_OK;
}

// ---- multi-device groups: queries sharded in contiguous blocks, index replicated, no collective (SURVEY 8e) -------------
bool is_group(const gtgpu_index* ix) { return ix && ix->replicas.size() > 1; }

int32_t count_group(gtgpu_index* ix, uint64_t n, const uint32_t* chr, const uint32_t* start, const uint32_t* end, int32_t min_overlap,
                    int mode, void* out, size_t elem) {
    if (!ix || (n && (!chr || !start || !end || !out))) return fail(GTGPU_ERR_INVALID, "count: null argument");
    std::lock_guard<std::mutex> glk(ix->ctx->group_mu);
    const size_t D = ix->replicas.size();
    return for_each_device(D, [&](size_t r) -> int32_t {
        uint64_t lo, hi;
        block_range(n, D, r, &lo, &hi);
        if (hi == lo) return GTGPU_OK;
        return count_host(ix->replicas[r], hi - lo, chr + lo, start + lo, end + lo, min_overlap, mode, (char*)out + lo * elem, elem);
    });
}

// Concatenates per-shard results (library-owned pinned buffers) into one buffer of the group's first device.
int32_t merge_bufs(gtgpu_ctx* ctx0, const std::vector<BufPtr>& parts, gtgpu_buf** out) {
    uint64_t total = 0;
    for (auto& p : parts) total += p ? p->len : 0;
    cudaSetDevice(ctx0->device);
    BufPtr buf;
    GT_TRY(buf_new(ctx0, total, 4, &buf));
    std::vector<uint64_t> base(parts.size() + 1, 0);
    for (size_t r = 0; r < parts.size(); ++r) base[r + 1] = base[r] + (parts[r] ? parts[r]->len : 0);
    for_each_device(parts.size(), [&](size_t r) -> int32_t {
        if (parts[r] && parts[r]->len) memcpy((uint32_t*)buf->block.ptr + base[r], parts[r]->block.ptr, parts[r]->len * 4);
        return GTGPU_OK;
    });
    *out = buf.release();
    return GTGPU_OK;
}

int32_t find_group(gtgpu_index* ix, uint64_t n, const uint32_t* chr, const uint32_t* start, const uint32_t* end, int32_t min_overlap,
                   uint64_t* out_offsets, gtgpu_buf** out_vals) {
    std::lock_guard<std::mutex> glk(ix->ctx->group_mu);
    const size_t D = ix->replicas.size();
    std::vector<BufPtr> parts(D);
    std::vector<std::vector<uint64_t>> offs(D);
    int32_t s = for_each_device(D, [&](size_t r) -> int32_t {
        uint64_t lo, hi;
        block_range(n, D, r, &lo, &hi);
        offs[r].assign(hi - lo + 1, 0);
        return find_host(ix->replicas[r], hi - lo, chr + lo, start + lo, end + lo, min_overlap, offs[r].data(), false, 0, nullptr, 0,
                         nullptr, &parts[r]);
    });
    if (s == GTGPU_OK) s = merge_bufs(ix->ctx, parts, out_vals);
    if (s == GTGPU_OK) {
        uint64_t base = 0;
        for (size_t r = 0; r < D; ++r) {
            uint64_t lo, hi;
            block_range(n, D, r, &lo, &hi);
            for (uint64_t i = 0; i < hi - lo; ++i) out_offsets[lo + i] = base + offs[r][i];
            base += offs[r][hi - lo];
        }
        out_offsets[n] = base;
    }
    return s;
}

// Tokenize on a group without the chunk pipeline (mid-sized batches and the pipeline's rare fallbacks): whole files are
// dealt to the devices in contiguous blocks, every device runs the plain path, results concatenate in device order.
int32_t tokenize_files_group_simple(gtgpu_index* ix, uint64_t n_files, const uint64_t* file_offsets, const uint32_t* chr,
                                    const uint32_t* start, const uint32_t* end, uint32_t unk_id, uint64_t* out_file_tok,
                                    gtgpu_buf** out_ids) {
    const size_t D = ix->replicas.size();
    std::vector<BufPtr> parts(D);
    std::vector<std::vector<uint64_t>> fo(D), tok(D);
    int32_t s = for_each_device(D, [&](size_t r) -> int32_t {
        uint64_t f0, f1;
        block_range(n_files, D, r, &f0, &f1);
        const uint64_t q0 = file_offsets[f0];
        fo[r].resize(f1 - f0 + 1);
        for (uint64_t f = f0; f <= f1; ++f) fo[r][f - f0] = file_offsets[f] - q0;
        tok[r].assign(f1 - f0 + 1, 0);
        return find_host(ix->replicas[r], file_offsets[f1] - q0, chr + q0, start + q0, end + q0, 0, nullptr, true, f1 - f0, fo[r].data(),
                         unk_id, tok[r].data(), &parts[r]);
    });
    if (s == GTGPU_OK) s = merge_bufs(ix->ctx, parts, out_ids);
    if (s == GTGPU_OK) {
        uint64_t base = 0;
        for (size_t r = 0; r < D; ++r) {
            uint64_t f0, f1;
            block_range(n_files, D, r, &f0, &f1);
            for (uint64_t f = f0; f < f1; ++f) out_file_tok[f] = base + tok[r][f - f0];
            base += tok[r][f1 - f0];
        }
        out_file_tok[n_files] = base;
    }
    return s;
}

// the non-pipelined path: one device, or whole files dealt to the devices of a group once the batch is worth it
int32_t tokenize_files_plain(gtgpu_index* ix, uint64_t n, uint64_t n_files, const uint64_t* file_offsets, const uint32_t* chr,
                             const uint32_t* start, const uint32_t* end, uint32_t unk_id, uint64_t* out_file_tok, gtgpu_buf** out_ids) {
    if (is_group(ix) && n >= (1u << 20) && n_files >= ix->replicas.size())
        return tokenize_files_group_simple(ix, n_files, file_offsets, chr, start, end, unk_id, out_file_tok, out_ids);
    BufPtr ids;
    GT_TRY(find_host(ix, n, chr, start, end, 0, nullptr, true, n_files, file_offsets, unk_id, out_file_tok, &ids));
    *out_ids = ids.release();
    return GTGPU_OK;
}

// queries per pipeline chunk (a multiple of the tile size): 32 M on one device; a group wants at least ~4 chunks per device
uint64_t pipe_chunk(const gtgpu_index* ix, uint64_t n) {
    uint64_t chunk = 32ull << 20;
    const uint64_t D = std::max<size_t>(ix->replicas.size(), 1);
    if (D > 1) chunk = std::min<uint64_t>(chunk, std::max<uint64_t>(n / (4 * D), 1ull << 20)) / FUSED_TILE * FUSED_TILE;
    if (const char* env = getenv("GTGPU_PIPE_CHUNK")) chunk = strtoull(env, nullptr, 10) / FUSED_TILE * FUSED_TILE;
    return chunk;
}
bool pipe_wanted(uint64_t n, uint64_t chunk) { return chunk >= (uint64_t)FUSED_TILE && n > chunk && (n + chunk - 1) / chunk <= 56; }

// gtgpu_tokenize_files for large batches: the queries stream through two device buffers per device in chunks, so the H2D
// copy of chunk k+1, the fused kernel of chunk k and the D2H copy of chunk k-1's ids overlap (PCIe is full duplex and the
// kernel is ~20x faster than either copy).  On a multi-device group the chunks are dealt round-robin to the devices
// (chunk k runs on device k mod D), so every device's copies and kernels overlap with every other's, and each chunk's ids
// go straight to their final place in ONE pinned result buffer: the host keeps the running total of all earlier chunks
// (8 bytes come back per chunk), so the result is bit-identical to a single launch on one device, whatever D is.
// Returns 1 in *fallback (and no result) for the rare cases the simple path handles: output larger than the
// optimistic capacity, a file with no token at all ([unk] insertion shifts the ids), or a tile overflow.
struct PipeDev {
    gtgpu_index* ix = nullptr;
    gtgpu_ctx* ctx = nullptr;
    uint32_t* in[2][3] = {{nullptr, nullptr, nullptr}, {nullptr, nullptr, nullptr}};
    uint16_t* d_w16[2] = {nullptr, nullptr};
    uint32_t* d_anc[2] = {nullptr, nullptr};
    uint32_t *d_ids = nullptr, *d_run_chr = nullptr, *d_wide_end = nullptr, *d_exc_start = nullptr;
    uint64_t *d_fo = nullptr, *d_raw_tok = nullptr, *d_chain = nullptr, *d_misc = nullptr, *d_run_off = nullptr, *d_wide_idx = nullptr;
    void* d_ws = nullptr;
    uint64_t cap = 0, n_local = 0;
    cudaEvent_t ev_in[2] = {nullptr, nullptr}, ev_free[2] = {nullptr, nullptr};
    std::unique_lock<std::mutex> lock;
};

int32_t tokenize_files_pipelined(gtgpu_index* gix, uint64_t n, uint64_t n_files, const uint64_t* file_offsets,
                                 const uint32_t* chr, const uint32_t* start, const uint32_t* end, uint64_t chunk,
                                 uint64_t* out_file_tok, gtgpu_buf** out_ids, int* fallback, uint64_t n_runs = 0,
                                 const uint64_t* run_offsets = nullptr, const uint32_t* run_chr = nullptr,
                                 const uint16_t* width16 = nullptr, uint64_t n_wide = 0, const uint64_t* wide_index = nullptr,
                                 const uint32_t* wide_end = nullptr, const uint32_t* packed = nullptr,
                                 const uint32_t* anchors = nullptr, uint32_t width_bits = 0, const uint32_t* exc_start = nullptr) {
    // packed != nullptr: the packed wire format (start / end rebuilt on the device from packed words + block anchors; the
    // exception list is (wide_index, exc_start, wide_end)); `start`, `end` and `width16` are then unused
    *fallback = 0;
    const uint64_t n_chunks = (n + chunk - 1) / chunk;
    const size_t D = std::max<size_t>(gix->replicas.size(), 1);
    const uint64_t cap_total = n + n / 4 + 1024;
    std::vector<PipeDev> devs(D);
    std::vector<cudaEvent_t> ev_done(n_chunks, nullptr);
    gtgpu_ctx* ctx0 = gix->ctx;

    // every file boundary belongs to the chunk that holds its first query; offsets are rebased to that chunk
    std::vector<uint64_t> rebased(n_files + 1), first_f(n_chunks + 1, 0);
    {
        uint64_t f = 0;
        for (uint64_t k = 0; k < n_chunks; ++k) {
            first_f[k] = f;
            const uint64_t q0 = k * chunk, q1 = std::min(n, q0 + chunk);
            while (f <= n_files && (file_offsets[f] < q1 || k + 1 == n_chunks)) {
                rebased[f] = file_offsets[f] - q0;
                ++f;
            }
        }
        first_f[n_chunks] = n_files + 1;
    }

    int32_t status = GTGPU_OK;
    cudaError_t cerr = cudaSuccess;
    BufPtr buf;
    uint64_t* h_raw_tok = nullptr;  // pinned: every chunk's slice of raw per-file id offsets (device-local numbering)
    auto cleanup = [&]() {
        for (auto& d : devs) {
            if (!d.ctx) continue;
            cudaSetDevice(d.ctx->device);
            cudaStreamSynchronize(d.ctx->stream);
            cudaStreamSynchronize(d.ctx->copy_in);
            cudaStreamSynchronize(d.ctx->copy_out);
            for (int b = 0; b < 2; ++b) {
                if (d.ev_in[b]) cudaEventDestroy(d.ev_in[b]);
                if (d.ev_free[b]) cudaEventDestroy(d.ev_free[b]);
            }
        }
        for (uint64_t k = 0; k < n_chunks; ++k)
            if (ev_done[k]) {
                cudaSetDevice(devs[k % D].ctx->device);
                cudaEventDestroy(ev_done[k]);
            }
        if (h_raw_tok) cudaFreeHost(h_raw_tok);
        cudaSetDevice(ctx0->device);
    };
    auto setup = [&]() -> int32_t {
        for (size_t r = 0; r < D; ++r) {
            PipeDev& d = devs[r];
            d.ix = D > 1 ? gix->replicas[r] : gix;
            d.ctx = d.ix->ctx;
            d.lock = std::unique_lock<std::mutex>(d.ctx->mu);
            gtgpu_ctx* ctx = d.ctx;
            GT_CUDA(cudaSetDevice(ctx->device));
            cudaStream_t st = ctx->stream;
            d.n_local = n_chunks / D + (r < n_chunks % D ? 1 : 0);
            d.cap = d.n_local * chunk + d.n_local * chunk / 4 + 1024;
            const int roles[2][3] = {{SC_CHR, SC_START, SC_END}, {SC_IN2_CHR, SC_IN2_START, SC_IN2_END}};
            for (int b = 0; b < 2; ++b)
                for (int a = 0; a < 3; ++a) GT_TRY(ctx->scratch_get(roles[b][a], chunk * 4, (void**)&d.in[b][a]));
            GT_TRY(ctx->scratch_get(SC_OUT_IDS, d.cap * 4, (void**)&d.d_ids));
            GT_TRY(ctx->scratch_get(SC_FILE_OFFS, (n_files + 1) * 8, (void**)&d.d_fo));
            GT_TRY(ctx->scratch_get(SC_FILE_TOK, (n_files + 1) * 8, (void**)&d.d_raw_tok));
            GT_TRY(ctx->scratch_get(SC_COUNTS, (d.n_local + 1) * 8, (void**)&d.d_chain));
            GT_TRY(ctx->scratch_get(SC_MISC, 64, (void**)&d.d_misc));
            GT_TRY(ctx->scratch_get(SC_TILE_STATUS, fused_workspace_bytes(chunk), &d.d_ws));
            // chromosome ids given as runs: ship the runs once, expand them per chunk on the device (no per-query chr H2D)
            if (run_offsets) {
                GT_TRY(ctx->scratch_get(SC_IN3_CHR, (n_runs + 1) * 8, (void**)&d.d_run_off));
                GT_TRY(ctx->scratch_get(SC_IN3_START, (n_runs + 1) * 4, (void**)&d.d_run_chr));
                GT_CUDA(cudaMemcpyAsync(d.d_run_off, run_offsets, (n_runs + 1) * 8, cudaMemcpyHostToDevice, st));
                GT_CUDA(cudaMemcpyAsync(d.d_run_chr, run_chr, n_runs * 4, cudaMemcpyHostToDevice, st));
            }
            // ends given as 16-bit widths (+ an exception list): 2 bytes per query cross PCIe instead of 4
            if (packed) {
                GT_TRY(ctx->scratch_get(SC_BARCODE, chunk / 32 * 4 + 64, (void**)&d.d_anc[0]));
                GT_TRY(ctx->scratch_get(SC_SET_ID, chunk / 32 * 4 + 64, (void**)&d.d_anc[1]));
                if (n_wide) {
                    GT_TRY(ctx->scratch_get(SC_IN3_END, n_wide * 8, (void**)&d.d_wide_idx));
                    GT_TRY(ctx->scratch_get(SC_MATRIX, n_wide * 4, (void**)&d.d_wide_end));
                    GT_TRY(ctx->scratch_get(SC_OUT_OFFS, n_wide * 4, (void**)&d.d_exc_start));
                    GT_CUDA(cudaMemcpyAsync(d.d_wide_idx, wide_index, n_wide * 8, cudaMemcpyHostToDevice, st));
                    GT_CUDA(cudaMemcpyAsync(d.d_wide_end, wide_end, n_wide * 4, cudaMemcpyHostToDevice, st));
                    GT_CUDA(cudaMemcpyAsync(d.d_exc_start, exc_start, n_wide * 4, cudaMemcpyHostToDevice, st));
                }
            } else if (width16) {
                GT_TRY(ctx->scratch_get(SC_BARCODE, chunk * 2, (void**)&d.d_w16[0]));
                GT_TRY(ctx->scratch_get(SC_SET_ID, chunk * 2, (void**)&d.d_w16[1]));
                if (n_wide) {
                    GT_TRY(ctx->scratch_get(SC_IN3_END, n_wide * 8, (void**)&d.d_wide_idx));
                    GT_TRY(ctx->scratch_get(SC_MATRIX, n_wide * 4, (void**)&d.d_wide_end));
                    GT_CUDA(cudaMemcpyAsync(d.d_wide_idx, wide_index, n_wide * 8, cudaMemcpyHostToDevice, st));
                    GT_CUDA(cudaMemcpyAsync(d.d_wide_end, wide_end, n_wide * 4, cudaMemcpyHostToDevice, st));
                }
            }
            GT_CUDA(cudaMemcpyAsync(d.d_fo, rebased.data(), (n_files + 1) * 8, cudaMemcpyHostToDevice, st));
            GT_CUDA(cudaMemsetAsync(d.d_chain, 0, (d.n_local + 1) * 8, st));
            GT_CUDA(cudaMemsetAsync(d.d_misc, 0, 64, st));
            for (int b = 0; b < 2; ++b) {
                GT_CUDA(cudaEventCreateWithFlags(&d.ev_in[b], cudaEventDisableTiming));
                GT_CUDA(cudaEventCreateWithFlags(&d.ev_free[b], cudaEventDisableTiming));
            }
            ctx->h_scalars[0] = 0;
        }
        for (uint64_t k = 0; k < n_chunks; ++k) {
            GT_CUDA(cudaSetDevice(devs[k % D].ctx->device));
            GT_CUDA(cudaEventCreateWithFlags(&ev_done[k], cudaEventDisableTiming));
        }
        for (auto& d : devs) {  // the host arrays above may be pageable: the copies must have consumed them
            GT_CUDA(cudaSetDevice(d.ctx->device));
            GT_CUDA(cudaStreamSynchronize(d.ctx->stream));
        }
        GT_CUDA(cudaSetDevice(ctx0->device));
        GT_CUDA(cudaHostAlloc((void**)&h_raw_tok, (n_files + 2) * 8, cudaHostAllocDefault));
        return buf_new(ctx0, cap_total, 4, &buf);
    };
    status = setup();
    if (status != GTGPU_OK) {
        cleanup();
        return status;
    }
    uint32_t* h_ids = (uint32_t*)buf->block.ptr;
    std::vector<uint64_t> gbase(n_chunks + 1, 0), local_lo(n_chunks, 0);
    bool overflow = false;
    auto drain = [&](uint64_t j) {  // ids of chunk j: device -> their final place in the pinned result, on the copy-out stream
        if (cerr != cudaSuccess) return;
        PipeDev& d = devs[j % D];
        const uint64_t i = j / D;
        cudaSetDevice(d.ctx->device);
        cerr = cudaEventSynchronize(ev_done[j]);
        volatile uint64_t* h_chain = d.ctx->h_scalars;  // [i] = ids this device produced before its i-th chunk
        const uint64_t lo = h_chain[i], hi = h_chain[i + 1];
        local_lo[j] = lo;
        gbase[j + 1] = gbase[j] + (hi - lo);
        if (hi > d.cap || gbase[j + 1] > cap_total) overflow = true;
        if (cerr == cudaSuccess && !overflow && hi > lo)
            cerr = cudaMemcpyAsync(h_ids + gbase[j], d.d_ids + lo, (hi - lo) * 4, cudaMemcpyDeviceToHost, d.ctx->copy_out);
    };
    auto fold = [&](cudaError_t e) {
        if (cerr == cudaSuccess) cerr = e;
    };
    try {
        for (uint64_t k = 0; k < n_chunks && status == GTGPU_OK && cerr == cudaSuccess; ++k) {
            PipeDev& d = devs[k % D];
            gtgpu_ctx* ctx = d.ctx;
            cudaStream_t st = ctx->stream;
            const uint64_t i = k / D;
            const int b = (int)(i & 1);
            const uint64_t q0 = k * chunk, cn = std::min(chunk, n - q0);
            fold(cudaSetDevice(ctx->device));
            if (i >= 2) fold(cudaStreamWaitEvent(ctx->copy_in, d.ev_free[b], 0));
            if (!run_offsets) fold(cudaMemcpyAsync(d.in[b][0], chr + q0, cn * 4, cudaMemcpyHostToDevice, ctx->copy_in));
            if (packed) {  // q0 is a multiple of the tile size, so the chunk starts on an anchor block
                fold(cudaMemcpyAsync(d.in[b][1], packed + q0, cn * 4, cudaMemcpyHostToDevice, ctx->copy_in));
                fold(cudaMemcpyAsync(d.d_anc[b], anchors + q0 / 32, (cn + 31) / 32 * 4, cudaMemcpyHostToDevice, ctx->copy_in));
            } else {
                fold(cudaMemcpyAsync(d.in[b][1], start + q0, cn * 4, cudaMemcpyHostToDevice, ctx->copy_in));
                if (width16) fold(cudaMemcpyAsync(d.d_w16[b], width16 + q0, cn * 2, cudaMemcpyHostToDevice, ctx->copy_in));
                else fold(cudaMemcpyAsync(d.in[b][2], end + q0, cn * 4, cudaMemcpyHostToDevice, ctx->copy_in));
            }
            fold(cudaEventRecord(d.ev_in[b], ctx->copy_in));
            fold(cudaStreamWaitEvent(st, d.ev_in[b], 0));
            if (cerr != cudaSuccess) break;
            if (packed) {
                const uint64_t lo = std::lower_bound(wide_index, wide_index + n_wide, q0) - wide_index;
                const uint64_t hi = std::lower_bound(wide_index, wide_index + n_wide, q0 + cn) - wide_index;
                status = launch_expand_packed(ctx, cn, d.in[b][1], d.d_anc[b], width_bits, d.in[b][1], d.in[b][2], hi - lo, d.d_wide_idx + lo,
                                              d.d_exc_start + lo, d.d_wide_end + lo, q0);
            } else if (width16) {
                const uint64_t lo = std::lower_bound(wide_index, wide_index + n_wide, q0) - wide_index;
                const uint64_t hi = std::lower_bound(wide_index, wide_index + n_wide, q0 + cn) - wide_index;
                status = launch_expand_widths(ctx, cn, d.in[b][1], d.d_w16[b], d.in[b][2], hi - lo, d.d_wide_idx + lo, d.d_wide_end + lo, q0);
            }
            if (run_offsets && status == GTGPU_OK) status = launch_expand_runs(ctx, n_runs, d.d_run_off, d.d_run_chr, q0, cn, d.in[b][0]);
            const uint64_t L = first_f[k + 1] - first_f[k];  // file boundaries owned by this chunk
            if (status == GTGPU_OK)
                status = launch_fused_find(d.ix, cn, L ? L - 1 : 0, d.d_fo + first_f[k], d.in[b][0], d.in[b][1], d.in[b][2], 0, d.d_ids, d.cap,
                                           nullptr, L ? d.d_raw_tok + first_f[k] : nullptr, d.d_ws, d.d_chain + i, d.d_chain + i + 1,
                                           (uint32_t*)(d.d_misc + 2));
            fold(cudaEventRecord(d.ev_free[b], st));
            fold(cudaMemcpyAsync((void*)(ctx->h_scalars + i + 1), d.d_chain + i + 1, 8, cudaMemcpyDeviceToHost, st));
            if (L) fold(cudaMemcpyAsync(h_raw_tok + first_f[k], d.d_raw_tok + first_f[k], L * 8, cudaMemcpyDeviceToHost, st));
            fold(cudaEventRecord(ev_done[k], st));
            if (k >= D) drain(k - D);  // one chunk per device stays in flight
        }
        if (status == GTGPU_OK)
            for (uint64_t j = n_chunks > D ? n_chunks - D : 0; j < n_chunks; ++j) drain(j);
    } catch (...) {
        cleanup();  // the copies into buf end before it goes back to the cache
        throw;
    }
    uint64_t total = 0, n_empty = 0;
    if (status == GTGPU_OK && cerr == cudaSuccess && !overflow) {
        for (auto& d : devs) {
            fold(cudaSetDevice(d.ctx->device));
            fold(cudaMemcpyAsync((void*)(d.ctx->h_scalars + 60), d.d_misc, 24, cudaMemcpyDeviceToHost, d.ctx->stream));
            fold(cudaStreamSynchronize(d.ctx->stream));
            fold(cudaStreamSynchronize(d.ctx->copy_out));
            if ((uint32_t)d.ctx->h_scalars[62] != 0) overflow = true;  // more than 2^32 hits inside one tile
        }
        total = gbase[n_chunks];
        if (cerr == cudaSuccess && !overflow) {
            // raw per-file offsets were numbered from each device's own running total: rebase them to the global one, then
            // apply the per-call [unk] rule (tokenizer.rs:158-160) — here only to detect files without ids
            for (uint64_t k = 0; k < n_chunks; ++k) {
                const uint64_t delta = gbase[k] - local_lo[k];
                for (uint64_t f = first_f[k]; f < first_f[k + 1]; ++f) out_file_tok[f] = h_raw_tok[f] + delta;
            }
            for (uint64_t f = 0; f < n_files; ++f) n_empty += out_file_tok[f + 1] == out_file_tok[f];
        }
    }
    cleanup();
    if (status != GTGPU_OK || cerr != cudaSuccess || overflow || n_empty > 0) {
        if (status != GTGPU_OK) return status;
        if (cerr != cudaSuccess) return fail(GTGPU_ERR_CUDA, std::string("tokenize_files (pipelined): ") + cudaGetErrorString(cerr));
        *fallback = 1;
        return GTGPU_OK;
    }
    buf->len = total;
    *out_ids = buf.release();
    return GTGPU_OK;
}

}  // namespace

extern "C" {

int32_t gtgpu_count(gtgpu_index* ix, uint64_t n, const uint32_t* chr, const uint32_t* start, const uint32_t* end,
                    int32_t min_overlap, uint32_t* out_counts) try {
    if (is_group(ix)) return count_group(ix, n, chr, start, end, min_overlap, COUNT_U32, out_counts, 4);
    return count_host(ix, n, chr, start, end, min_overlap, COUNT_U32, out_counts, 4);
} GT_CATCH

int32_t gtgpu_bits_count(gtgpu_index* ix, uint64_t n, const uint32_t* chr, const uint32_t* start,
                         const uint32_t* end, uint64_t* out_counts) try {
    if (is_group(ix)) return count_group(ix, n, chr, start, end, 0, COUNT_BITS_RAW_U64, out_counts, 8);
    return count_host(ix, n, chr, start, end, 0, COUNT_BITS_RAW_U64, out_counts, 8);
} GT_CATCH

int32_t gtgpu_any(gtgpu_index* ix, uint64_t n, const uint32_t* chr, const uint32_t* start, const uint32_t* end,
                  int32_t min_overlap, uint8_t* out_any) try {
    if (is_group(ix)) return count_group(ix, n, chr, start, end, min_overlap, COUNT_ANY_U8, out_any, 1);
    return count_host(ix, n, chr, start, end, min_overlap, COUNT_ANY_U8, out_any, 1);
} GT_CATCH

int32_t gtgpu_find(gtgpu_index* ix, uint64_t n, const uint32_t* chr, const uint32_t* start, const uint32_t* end,
                   int32_t min_overlap, uint64_t* out_offsets, gtgpu_buf** out_vals) try {
    if (!ix || !out_offsets || !out_vals || (n && (!chr || !start || !end)))
        return fail(GTGPU_ERR_INVALID, "find: null argument");
    if (is_group(ix) && n >= (1u << 16)) return find_group(ix, n, chr, start, end, min_overlap, out_offsets, out_vals);
    BufPtr vals;
    GT_TRY(find_host(ix, n, chr, start, end, min_overlap, out_offsets, false, 0, nullptr, 0, nullptr, &vals));
    *out_vals = vals.release();
    return GTGPU_OK;
} GT_CATCH

int32_t gtgpu_tokenize_files(gtgpu_index* ix, uint64_t n_files, const uint64_t* file_offsets, const uint32_t* chr,
                             const uint32_t* start, const uint32_t* end, uint32_t unk_id,
                             uint64_t* out_file_token_offsets, gtgpu_buf** out_ids) try {
    if (!ix || !file_offsets || !out_file_token_offsets || !out_ids)
        return fail(GTGPU_ERR_INVALID, "tokenize_files: null argument");
    if (file_offsets[0] != 0) return fail(GTGPU_ERR_INVALID, "tokenize_files: file_offsets[0] must be 0");
    for (uint64_t f = 0; f < n_files; ++f)
        if (file_offsets[f] > file_offsets[f + 1])
            return fail(GTGPU_ERR_INVALID, "tokenize_files: file_offsets not monotone");
    uint64_t n = file_offsets[n_files];
    if (n && (!chr || !start || !end)) return fail(GTGPU_ERR_INVALID, "tokenize_files: null query arrays");
    std::unique_lock<std::mutex> glk;
    if (is_group(ix)) glk = std::unique_lock<std::mutex>(ix->ctx->group_mu);
    const uint64_t chunk = pipe_chunk(ix, n);
    if (pipe_wanted(n, chunk)) {
        int fallback = 0;
        GT_TRY(tokenize_files_pipelined(ix, n, n_files, file_offsets, chr, start, end, chunk, out_file_token_offsets, out_ids,
                                        &fallback));
        if (!fallback) return GTGPU_OK;
    }
    return tokenize_files_plain(ix, n, n_files, file_offsets, chr, start, end, unk_id, out_file_token_offsets, out_ids);
} GT_CATCH

int32_t gtgpu_tokenize_files_runs(gtgpu_index* ix, uint64_t n_files, const uint64_t* file_offsets, uint64_t n_runs,
                                  const uint64_t* run_offsets, const uint32_t* run_chr, const uint32_t* start,
                                  const uint32_t* end, uint32_t unk_id, uint64_t* out_file_token_offsets,
                                  gtgpu_buf** out_ids) try {
    if (!ix || !file_offsets || !run_offsets || !out_file_token_offsets || !out_ids || (n_runs && !run_chr))
        return fail(GTGPU_ERR_INVALID, "tokenize_files_runs: null argument");
    if (file_offsets[0] != 0 || run_offsets[0] != 0)
        return fail(GTGPU_ERR_INVALID, "tokenize_files_runs: offsets must start at 0");
    for (uint64_t f = 0; f < n_files; ++f)
        if (file_offsets[f] > file_offsets[f + 1]) return fail(GTGPU_ERR_INVALID, "tokenize_files_runs: file_offsets not monotone");
    for (uint64_t r = 0; r < n_runs; ++r)
        if (run_offsets[r] > run_offsets[r + 1]) return fail(GTGPU_ERR_INVALID, "tokenize_files_runs: run_offsets not monotone");
    const uint64_t n = file_offsets[n_files];
    if (run_offsets[n_runs] != n) return fail(GTGPU_ERR_INVALID, "tokenize_files_runs: runs do not cover the queries");
    if (n && (!start || !end)) return fail(GTGPU_ERR_INVALID, "tokenize_files_runs: null query arrays");
    std::unique_lock<std::mutex> glk;
    if (is_group(ix)) glk = std::unique_lock<std::mutex>(ix->ctx->group_mu);
    const uint64_t chunk = pipe_chunk(ix, n);
    if (pipe_wanted(n, chunk)) {
        int fallback = 0;
        GT_TRY(tokenize_files_pipelined(ix, n, n_files, file_offsets, nullptr, start, end, chunk, out_file_token_offsets, out_ids,
                                        &fallback, n_runs, run_offsets, run_chr));
        if (!fallback) return GTGPU_OK;
    }
    // small batches and the rare fallbacks: expand on the host and take the plain path
    std::vector<uint32_t> chr(n);
    for (uint64_t r = 0; r < n_runs; ++r) std::fill(chr.begin() + run_offsets[r], chr.begin() + run_offsets[r + 1], run_chr[r]);
    return tokenize_files_plain(ix, n, n_files, file_offsets, chr.data(), start, end, unk_id, out_file_token_offsets, out_ids);
} GT_CATCH

int32_t gtgpu_tokenize_files_compact(gtgpu_index* ix, uint64_t n_files, const uint64_t* file_offsets, uint64_t n_runs,
                                     const uint64_t* run_offsets, const uint32_t* run_chr, const uint32_t* start,
                                     const uint16_t* width16, uint64_t n_wide, const uint64_t* wide_index,
                                     const uint32_t* wide_end, uint32_t unk_id, uint64_t* out_file_token_offsets,
                                     gtgpu_buf** out_ids) try {
    if (!ix || !file_offsets || !run_offsets || !out_file_token_offsets || !out_ids || (n_runs && !run_chr) ||
        (n_wide && (!wide_index || !wide_end)))
        return fail(GTGPU_ERR_INVALID, "tokenize_files_compact: null argument");
    if (file_offsets[0] != 0 || run_offsets[0] != 0)
        return fail(GTGPU_ERR_INVALID, "tokenize_files_compact: offsets must start at 0");
    for (uint64_t f = 0; f < n_files; ++f)
        if (file_offsets[f] > file_offsets[f + 1]) return fail(GTGPU_ERR_INVALID, "tokenize_files_compact: file_offsets not monotone");
    for (uint64_t r = 0; r < n_runs; ++r)
        if (run_offsets[r] > run_offsets[r + 1]) return fail(GTGPU_ERR_INVALID, "tokenize_files_compact: run_offsets not monotone");
    const uint64_t n = file_offsets[n_files];
    if (run_offsets[n_runs] != n) return fail(GTGPU_ERR_INVALID, "tokenize_files_compact: runs do not cover the queries");
    if (n && (!start || !width16)) return fail(GTGPU_ERR_INVALID, "tokenize_files_compact: null query arrays");
    for (uint64_t i = 0; i < n_wide; ++i)
        if (wide_index[i] >= n || (i && wide_index[i] <= wide_index[i - 1]))
            return fail(GTGPU_ERR_INVALID, "tokenize_files_compact: wide_index must be strictly increasing and < n");
    std::unique_lock<std::mutex> glk;
    if (is_group(ix)) glk = std::unique_lock<std::mutex>(ix->ctx->group_mu);
    const uint64_t chunk = pipe_chunk(ix, n);
    if (pipe_wanted(n, chunk)) {
        int fallback = 0;
        GT_TRY(tokenize_files_pipelined(ix, n, n_files, file_offsets, nullptr, start, nullptr, chunk, out_file_token_offsets, out_ids,
                                        &fallback, n_runs, run_offsets, run_chr, width16, n_wide, wide_index, wide_end));
        if (!fallback) return GTGPU_OK;
    }
    // small batches and the rare fallbacks: expand on the host and take the plain path
    std::vector<uint32_t> chr(n), end(n);
    for (uint64_t r = 0; r < n_runs; ++r) std::fill(chr.begin() + run_offsets[r], chr.begin() + run_offsets[r + 1], run_chr[r]);
    for (uint64_t i = 0; i < n; ++i) end[i] = start[i] + width16[i];
    for (uint64_t i = 0; i < n_wide; ++i) end[wide_index[i]] = wide_end[i];
    return tokenize_files_plain(ix, n, n_files, file_offsets, chr.data(), start, end.data(), unk_id, out_file_token_offsets, out_ids);
} GT_CATCH

int32_t gtgpu_tokenize_files_packed(gtgpu_index* ix, uint64_t n_files, const uint64_t* file_offsets, uint64_t n_runs,
                                    const uint64_t* run_offsets, const uint32_t* run_chr, uint32_t width_bits, const uint32_t* packed,
                                    const uint32_t* anchors, uint64_t n_exc, const uint64_t* exc_index, const uint32_t* exc_start,
                                    const uint32_t* exc_end, uint32_t unk_id, uint64_t* out_file_token_offsets,
                                    gtgpu_buf** out_ids) try {
    if (!ix || !file_offsets || !run_offsets || !out_file_token_offsets || !out_ids || (n_runs && !run_chr) ||
        (n_exc && (!exc_index || !exc_start || !exc_end)))
        return fail(GTGPU_ERR_INVALID, "tokenize_files_packed: null argument");
    if (width_bits < 1 || width_bits > 24) return fail(GTGPU_ERR_INVALID, "tokenize_files_packed: width_bits must be 1..24");
    if (file_offsets[0] != 0 || run_offsets[0] != 0)
        return fail(GTGPU_ERR_INVALID, "tokenize_files_packed: offsets must start at 0");
    for (uint64_t f = 0; f < n_files; ++f)
        if (file_offsets[f] > file_offsets[f + 1]) return fail(GTGPU_ERR_INVALID, "tokenize_files_packed: file_offsets not monotone");
    for (uint64_t r = 0; r < n_runs; ++r)
        if (run_offsets[r] > run_offsets[r + 1]) return fail(GTGPU_ERR_INVALID, "tokenize_files_packed: run_offsets not monotone");
    const uint64_t n = file_offsets[n_files];
    if (run_offsets[n_runs] != n) return fail(GTGPU_ERR_INVALID, "tokenize_files_packed: runs do not cover the queries");
    if (n && (!packed || !anchors)) return fail(GTGPU_ERR_INVALID, "tokenize_files_packed: null query arrays");
    for (uint64_t i = 0; i < n_exc; ++i)
        if (exc_index[i] >= n || (i && exc_index[i] <= exc_index[i - 1]))
            return fail(GTGPU_ERR_INVALID, "tokenize_files_packed: exc_index must be strictly increasing and < n");
    std::unique_lock<std::mutex> glk;
    if (is_group(ix)) glk = std::unique_lock<std::mutex>(ix->ctx->group_mu);
    const uint64_t chunk = pipe_chunk(ix, n);
    if (pipe_wanted(n, chunk)) {
        int fallback = 0;
        GT_TRY(tokenize_files_pipelined(ix, n, n_files, file_offsets, nullptr, nullptr, nullptr, chunk, out_file_token_offsets, out_ids,
                                        &fallback, n_runs, run_offsets, run_chr, nullptr, n_exc, exc_index, exc_end, packed, anchors,
                                        width_bits, exc_start));
        if (!fallback) return GTGPU_OK;
    }
    // small batches and the rare fallbacks: expand on the host and take the plain path
    std::vector<uint32_t> chr(n), start(n), end(n);
    for (uint64_t r = 0; r < n_runs; ++r) std::fill(chr.begin() + run_offsets[r], chr.begin() + run_offsets[r + 1], run_chr[r]);
    const uint32_t off_bits = 32 - width_bits, off_mask = (1u << off_bits) - 1u;
    for (uint64_t i = 0; i < n; ++i) {
        start[i] = anchors[i >> 5] + (packed[i] & off_mask);
        end[i] = start[i] + (packed[i] >> off_bits);
    }
    for (uint64_t i = 0; i < n_exc; ++i) {
        start[exc_index[i]] = exc_start[i];
        end[exc_index[i]] = exc_end[i];
    }
    return tokenize_files_plain(ix, n, n_files, file_offsets, chr.data(), start.data(), end.data(), unk_id, out_file_token_offsets,
                                out_ids);
} GT_CATCH

int32_t gtgpu_count_dev(gtgpu_index* ix, uint64_t n, const uint32_t* d_chr, const uint32_t* d_start,
                        const uint32_t* d_end, int32_t min_overlap, uint32_t* d_out_counts) try {
    if (!ix || (n && (!d_chr || !d_start || !d_end || !d_out_counts)))
        return fail(GTGPU_ERR_INVALID, "count_dev: null argument");
    std::lock_guard<std::mutex> lk(ix->ctx->mu);
    GT_CUDA(cudaSetDevice(ix->ctx->device));
    return launch_count(ix, n, d_chr, d_start, d_end, min_overlap, COUNT_U32, d_out_counts);
} GT_CATCH

int32_t gtgpu_find_dev(gtgpu_index* ix, uint64_t n, const uint32_t* d_chr, const uint32_t* d_start,
                       const uint32_t* d_end, int32_t min_overlap, uint64_t n_files, const uint64_t* d_file_offsets,
                       uint32_t* d_out_ids, uint64_t ids_capacity, uint64_t* d_out_offsets,
                       uint64_t* d_out_file_token_offsets, uint64_t* d_out_total) try {
    if (!ix || !d_out_total || (n && (!d_chr || !d_start || !d_end)) || (ids_capacity && !d_out_ids))
        return fail(GTGPU_ERR_INVALID, "find_dev: null argument");
    if (d_out_file_token_offsets && !d_file_offsets)
        return fail(GTGPU_ERR_INVALID, "find_dev: per-file offsets requested without d_file_offsets");
    gtgpu_ctx* ctx = ix->ctx;
    std::lock_guard<std::mutex> lk(ctx->mu);
    GT_CUDA(cudaSetDevice(ctx->device));
    void* d_ws = nullptr;
    GT_TRY(ctx->scratch_get(SC_TILE_STATUS, fused_workspace_bytes(n), &d_ws));
    uint64_t* d_misc = nullptr;
    GT_TRY(ctx->scratch_get(SC_MISC, 64, (void**)&d_misc));
    GT_CUDA(cudaMemsetAsync(d_misc, 0, 64, ctx->stream));
    return launch_fused_find(ix, n, d_out_file_token_offsets ? n_files : 0, d_file_offsets, d_chr, d_start, d_end,
                             min_overlap, d_out_ids, ids_capacity, d_out_offsets, d_out_file_token_offsets, d_ws, nullptr,
                             d_out_total, (uint32_t*)(d_misc + 2));
} GT_CATCH

int32_t gtgpu_unk_rule_dev(gtgpu_ctx* ctx, uint64_t n_files, const uint64_t* d_raw_file_token_offsets,
                           const uint32_t* d_raw_ids, uint32_t unk_id, uint64_t* d_out_file_token_offsets,
                           uint32_t* d_out_ids, uint64_t* d_out_n_empty) try {
    if (!ctx || !d_raw_file_token_offsets || !d_out_file_token_offsets || !d_out_ids || !d_out_n_empty)
        return fail(GTGPU_ERR_INVALID, "unk_rule_dev: null argument");
    std::lock_guard<std::mutex> lk(ctx->mu);
    GT_CUDA(cudaSetDevice(ctx->device));
    GT_TRY(launch_unk_offsets(ctx, n_files, d_raw_file_token_offsets, d_out_file_token_offsets, d_out_n_empty));
    return launch_unk_expand(ctx, n_files, d_raw_file_token_offsets, d_out_file_token_offsets, d_raw_ids, unk_id,
                             d_out_ids);
} GT_CATCH

}  // extern "C"
