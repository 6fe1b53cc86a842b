// scoring.cu — gtars-scoring on the device: fragments x consensus-peak count matrices.
//
//   gtgpu_score_matrix    region_scoring_from_fragments   (gtars-scoring/src/fragment_scoring.rs:19-121)
//   gtgpu_score_barcodes  barcode_scoring_from_fragments  (fragment_scoring.rs:126-155)
//
// Both are the find kernel with a different reducer.  Atac mode turns every fragment into two queries — the shifted
// start [s+4, s+5) and the reversed end interval (start = e-5, end = e-6, exactly as fragment_scoring.rs:79-84 builds
// it; the find kernel resolves start >= end queries through the reference-faithful walk) — Chip mode uses the fragment
// itself.  Device plan:
//   matrix:   queries -> fused find with per-file id offsets -> histogram of (file, id) with 32-bit atomics
//   barcodes: fused find with per-fragment offsets -> barcode of every hit -> two stable radix sorts (peak, then
//             barcode) -> run-length encode -> CSR (barcode offsets, peaks, counts)
#include <algorithm>

#include "common.cuh"

namespace gtgpu {

// fragment i -> queries 2i (start side) and 2i+1 (end side); u32 arithmetic wraps like the reference's release build
__global__ void score_atac_queries_kernel(uint64_t n, const uint32_t* __restrict__ chr, const uint32_t* __restrict__ start,
                                          const uint32_t* __restrict__ end, uint32_t* __restrict__ qc,
                                          uint32_t* __restrict__ qs, uint32_t* __restrict__ qe) {
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        const uint32_t c = chr[i], ns = start[i] + 4u, ne = end[i] - 5u;
        reinterpret_cast<uint2*>(qc)[i] = make_uint2(c, c);
        reinterpret_cast<uint2*>(qs)[i] = make_uint2(ns, ne);
        reinterpret_cast<uint2*>(qe)[i] = make_uint2(ns + 1u, ne - 1u);
    }
}

__global__ void score_double_offsets_kernel(uint64_t count, const uint64_t* __restrict__ in, uint64_t* __restrict__ out) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < count) out[i] = 2 * in[i];
}

// hit h belongs to the file whose raw id range [file_tok[f], file_tok[f+1]) holds it
__global__ void score_hist_kernel(uint64_t n_hits, const uint32_t* __restrict__ ids, uint64_t n_files,
                                  const uint64_t* __restrict__ file_tok, uint64_t n_cols, uint32_t* __restrict__ mat) {
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t h = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; h < n_hits; h += stride) {
        uint64_t lo = 0, hi = n_files;  // last f with file_tok[f] <= h
        while (hi - lo > 1) {
            const uint64_t mid = (lo + hi) >> 1;
            if (__ldg(file_tok + mid) <= h) lo = mid;
            else hi = mid;
        }
        const uint32_t v = __ldcs(ids + h);
        if (v < n_cols) atomicAdd(mat + lo * n_cols + v, 1u);  // CountMatrix::increment is bounds-checked (counts.rs:49-56)
    }
}

__global__ void score_hit_barcodes_kernel(uint64_t n, const uint64_t* __restrict__ offsets, const uint32_t* __restrict__ barcode,
                                          uint32_t* __restrict__ hit_bc) {
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        const uint32_t b = barcode[i];
        for (uint64_t j = offsets[i]; j < offsets[i + 1]; ++j) hit_bc[j] = b;
    }
}

// 1 where a new (barcode, peak) run starts
__global__ void score_run_heads_kernel(uint64_t n, const uint32_t* __restrict__ bc, const uint32_t* __restrict__ pk,
                                       unsigned long long* __restrict__ head) {
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t h = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; h < n; h += stride)
        head[h] = (h == 0 || bc[h] != bc[h - 1] || pk[h] != pk[h - 1]) ? 1ull : 0ull;
}

__global__ void score_run_starts_kernel(uint64_t n, const unsigned long long* __restrict__ head,
                                        const unsigned long long* __restrict__ rank, unsigned long long* __restrict__ run_start) {
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t h = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; h < n; h += stride)
        if (head[h]) run_start[rank[h]] = h;
}

__global__ void score_runs_out_kernel(uint64_t nnz, uint64_t n_hits, const unsigned long long* __restrict__ run_start,
                                      const uint32_t* __restrict__ pk, uint32_t* __restrict__ out_peak,
                                      uint32_t* __restrict__ out_count) {
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t u = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; u < nnz; u += stride) {
        const uint64_t a = run_start[u], b = u + 1 < nnz ? run_start[u + 1] : n_hits;
        out_peak[u] = pk[a];
        out_count[u] = (uint32_t)(b - a);
    }
}

// offsets[b] = number of runs whose barcode is < b
__global__ void score_barcode_offsets_kernel(uint32_t n_barcodes, uint64_t nnz, const unsigned long long* __restrict__ run_start,
                                             const uint32_t* __restrict__ bc, uint64_t* __restrict__ out) {
    const uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b > n_barcodes) return;
    uint64_t lo = 0, hi = nnz;
    while (lo < hi) {
        const uint64_t mid = (lo + hi) >> 1;
        if (bc[run_start[mid]] < b) lo = mid + 1;
        else hi = mid;
    }
    out[b] = lo;
}

static int grid_for(gtgpu_ctx* ctx, uint64_t n) {
    return (int)std::max<uint64_t>(1, std::min<uint64_t>((n + 255) / 256, (uint64_t)ctx->sm_count * 16));
}

static int bits_for(uint64_t n_values) {
    int bits = 1;
    while (bits < 32 && (1ull << bits) < n_values) ++bits;
    return bits;
}

// Shared front end: fused find over device-resident queries with the optimistic capacity + exact re-run protocol.
// Returns the raw ids in SC_OUT_IDS (*d_ids) and their number.
int32_t fused_find_all(gtgpu_index* ix, uint64_t nq, uint64_t n_files, const uint64_t* d_qfo, const uint32_t* d_qc,
                        const uint32_t* d_qs, const uint32_t* d_qe, uint64_t* d_offsets, uint64_t* d_file_tok,
                        uint32_t** d_ids, uint64_t* total_out) {
    gtgpu_ctx* ctx = ix->ctx;
    cudaStream_t st = ctx->stream;
    void* d_ws;
    uint64_t* d_misc;
    GT_TRY(ctx->scratch_get(SC_TILE_STATUS, fused_workspace_bytes(nq), &d_ws));
    GT_TRY(ctx->scratch_get(SC_MISC, 64, (void**)&d_misc));
    uint64_t cap = nq + nq / 4 + 1024, total = 0;
    for (int attempt = 0; attempt < 2; ++attempt) {
        GT_TRY(ctx->scratch_get(SC_OUT_IDS, cap * 4, (void**)d_ids));
        GT_CUDA(cudaMemsetAsync(d_misc, 0, 64, st));
        GT_TRY(launch_fused_find(ix, nq, n_files, d_qfo, d_qc, d_qs, d_qe, 0, *d_ids, cap, d_offsets, d_file_tok, d_ws, nullptr,
                                 d_misc, (uint32_t*)(d_misc + 2)));
        GT_CUDA(cudaMemcpyAsync(ctx->h_scalars, d_misc, 24, cudaMemcpyDeviceToHost, st));
        GT_CUDA(cudaStreamSynchronize(st));
        total = ctx->h_scalars[0];
        if ((uint32_t)ctx->h_scalars[2] != 0) return fail(GTGPU_ERR_UNSUPPORTED, "score: tile overflow");
        if (total <= cap) break;
        if (attempt == 1) return fail(GTGPU_ERR_CAPACITY, "score: output capacity exceeded twice");
        cap = total;
    }
    *total_out = total;
    return GTGPU_OK;
}

// Device-resident core of gtgpu_score_matrix: d_out_counts (n_files x n_cols u32) is zeroed here unless `accumulate`.
static int32_t score_matrix_dev_locked(gtgpu_index* ix, uint64_t n_files, const uint64_t* d_file_offsets, uint64_t n,
                                       const uint32_t* d_chr, const uint32_t* d_start, const uint32_t* d_end, int32_t mode,
                                       uint64_t n_cols, uint32_t* d_out_counts, bool accumulate = false) {
    gtgpu_ctx* ctx = ix->ctx;
    cudaStream_t st = ctx->stream;
    if (!accumulate) GT_CUDA(cudaMemsetAsync(d_out_counts, 0, n_files * n_cols * 4, st));
    if (n == 0 || n_files == 0 || n_cols == 0) return GTGPU_OK;
    const uint32_t *qc = d_chr, *qs = d_start, *qe = d_end;
    const uint64_t* qfo = d_file_offsets;
    uint64_t nq = n;
    if (mode == GTGPU_SCORE_ATAC) {
        uint32_t *c2, *s2, *e2;
        uint64_t* fo2;
        nq = 2 * n;
        GT_TRY(ctx->scratch_get(SC_IN2_CHR, nq * 4, (void**)&c2));
        GT_TRY(ctx->scratch_get(SC_IN2_START, nq * 4, (void**)&s2));
        GT_TRY(ctx->scratch_get(SC_IN2_END, nq * 4, (void**)&e2));
        GT_TRY(ctx->scratch_get(SC_FILE_TOK2, (n_files + 1) * 8, (void**)&fo2));
        score_atac_queries_kernel<<<grid_for(ctx, n), 256, 0, st>>>(n, d_chr, d_start, d_end, c2, s2, e2);
        score_double_offsets_kernel<<<(unsigned)((n_files + 1 + 255) / 256), 256, 0, st>>>(n_files + 1, d_file_offsets, fo2);
        ctx->launches += 2;
        qc = c2; qs = s2; qe = e2; qfo = fo2;
    }
    if (nq >= 0xFFFFFFFFull) return fail(GTGPU_ERR_UNSUPPORTED, "score_matrix: more than 2^32-2 queries per call");
    uint64_t* d_file_tok;
    GT_TRY(ctx->scratch_get(SC_FILE_TOK, (n_files + 1) * 8, (void**)&d_file_tok));
    uint32_t* d_ids = nullptr;
    uint64_t total = 0;
    GT_TRY(fused_find_all(ix, nq, n_files, qfo, qc, qs, qe, nullptr, d_file_tok, &d_ids, &total));
    if (total) {
        score_hist_kernel<<<grid_for(ctx, total), 256, 0, st>>>(total, d_ids, n_files, d_file_tok, n_cols, d_out_counts);
        ctx->launches++;
    }
    GT_CUDA(cudaGetLastError());
    return GTGPU_OK;
}

}  // namespace gtgpu

using namespace gtgpu;

extern "C" int32_t gtgpu_score_matrix_dev(gtgpu_index* ix, uint64_t n_files, const uint64_t* d_file_offsets, uint64_t n,
                                          const uint32_t* d_chr, const uint32_t* d_start, const uint32_t* d_end, int32_t mode,
                                          uint64_t n_cols, uint32_t* d_out_counts) try {
    if (!ix || !d_out_counts || !d_file_offsets || (n && (!d_chr || !d_start || !d_end)))
        return fail(GTGPU_ERR_INVALID, "score_matrix_dev: null argument");
    if (mode != GTGPU_SCORE_ATAC && mode != GTGPU_SCORE_CHIP) return fail(GTGPU_ERR_INVALID, "score_matrix_dev: unknown mode");
    gtgpu_ctx* ctx = ix->ctx;
    std::lock_guard<std::mutex> lk(ctx->mu);
    GT_CUDA(cudaSetDevice(ctx->device));
    return score_matrix_dev_locked(ix, n_files, d_file_offsets, n, d_chr, d_start, d_end, mode, n_cols, d_out_counts);
} GT_CATCH

static int32_t score_matrix_one(gtgpu_index* ix, uint64_t n_files, const uint64_t* file_offsets, uint64_t n,
                                      const uint32_t* chr, const uint32_t* start, const uint32_t* end, int32_t mode,
                                      uint64_t n_cols, uint32_t* out_counts) {
    if (!ix || !out_counts || !file_offsets || (n && (!chr || !start || !end)))
        return fail(GTGPU_ERR_INVALID, "score_matrix: null argument");
    if (mode != GTGPU_SCORE_ATAC && mode != GTGPU_SCORE_CHIP) return fail(GTGPU_ERR_INVALID, "score_matrix: unknown mode");
    if (file_offsets[0] != 0 || file_offsets[n_files] != n) return fail(GTGPU_ERR_INVALID, "score_matrix: file_offsets must span [0, n]");
    for (uint64_t f = 0; f < n_files; ++f)
        if (file_offsets[f] > file_offsets[f + 1]) return fail(GTGPU_ERR_INVALID, "score_matrix: file_offsets must not decrease");
    gtgpu_ctx* ctx = ix->ctx;
    std::lock_guard<std::mutex> lk(ctx->mu);
    GT_CUDA(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    uint32_t *d_chr, *d_start, *d_end, *d_mat;
    uint64_t* d_fo;
    GT_TRY(ctx->scratch_get(SC_CHR, n * 4, (void**)&d_chr));
    GT_TRY(ctx->scratch_get(SC_START, n * 4, (void**)&d_start));
    GT_TRY(ctx->scratch_get(SC_END, n * 4, (void**)&d_end));
    GT_TRY(ctx->scratch_get(SC_FILE_OFFS, (n_files + 1) * 8, (void**)&d_fo));
    GT_TRY(ctx->scratch_get(SC_MATRIX, std::max<uint64_t>(n_files * n_cols * 4, 4), (void**)&d_mat));
    if (n) {
        GT_CUDA(cudaMemcpyAsync(d_chr, chr, n * 4, cudaMemcpyHostToDevice, st));
        GT_CUDA(cudaMemcpyAsync(d_start, start, n * 4, cudaMemcpyHostToDevice, st));
        GT_CUDA(cudaMemcpyAsync(d_end, end, n * 4, cudaMemcpyHostToDevice, st));
    }
    GT_CUDA(cudaMemcpyAsync(d_fo, file_offsets, (n_files + 1) * 8, cudaMemcpyHostToDevice, st));
    GT_TRY(score_matrix_dev_locked(ix, n_files, d_fo, n, d_chr, d_start, d_end, mode, n_cols, d_mat));
    if (n_files * n_cols) GT_CUDA(cudaMemcpyAsync(out_counts, d_mat, n_files * n_cols * 4, cudaMemcpyDeviceToHost, st));
    GT_CUDA(cudaStreamSynchronize(st));
    return GTGPU_OK;
}


// Multi-device group: counts are additive, so the fragments are dealt to the devices in contiguous blocks (each with the
// file boundaries that fall inside its block), every device fills a full n_files x n_cols matrix and the host adds them.
extern "C" int32_t gtgpu_score_matrix(gtgpu_index* ix, uint64_t n_files, const uint64_t* file_offsets, uint64_t n,
                                      const uint32_t* chr, const uint32_t* start, const uint32_t* end, int32_t mode,
                                      uint64_t n_cols, uint32_t* out_counts) try {
    if (!ix || !out_counts || !file_offsets || (n && (!chr || !start || !end)))
        return fail(GTGPU_ERR_INVALID, "score_matrix: null argument");
    const size_t D = ix->replicas.size();
    if (D <= 1 || n < (1u << 20)) return score_matrix_one(ix, n_files, file_offsets, n, chr, start, end, mode, n_cols, out_counts);
    if (file_offsets[0] != 0 || file_offsets[n_files] != n) return fail(GTGPU_ERR_INVALID, "score_matrix: file_offsets must span [0, n]");
    for (uint64_t f = 0; f < n_files; ++f)
        if (file_offsets[f] > file_offsets[f + 1]) return fail(GTGPU_ERR_INVALID, "score_matrix: file_offsets must not decrease");
    std::lock_guard<std::mutex> glk(ix->ctx->group_mu);
    const uint64_t cells = n_files * n_cols;
    std::vector<std::vector<uint32_t>> partial(D);
    int32_t s = for_each_device(D, [&](size_t r) -> int32_t {
        uint64_t lo, hi;
        block_range(n, D, r, &lo, &hi);
        std::vector<uint64_t> fo(n_files + 1);
        for (uint64_t f = 0; f <= n_files; ++f) fo[f] = std::min(std::max(file_offsets[f], lo), hi) - lo;
        uint32_t* dst = r == 0 ? out_counts : (partial[r].resize(cells), partial[r].data());
        return score_matrix_one(ix->replicas[r], n_files, fo.data(), hi - lo, chr + lo, start + lo, end + lo, mode, n_cols, dst);
    });
    if (s != GTGPU_OK) return s;
    for_each_device(D, [&](size_t t) -> int32_t {  // D host threads, each a contiguous range of cells
        uint64_t c0, c1;
        block_range(cells, D, t, &c0, &c1);
        for (size_t r = 1; r < D; ++r)
            for (uint64_t c = c0; c < c1; ++c) out_counts[c] += partial[r][c];
        return GTGPU_OK;
    });
    return GTGPU_OK;
} GT_CATCH

// Device-resident core of gtgpu_score_barcodes (the caller holds ctx->mu): fragments and dense barcode ids on the device,
// out_barcode_offsets (n_barcodes + 1) on the host.
static int32_t score_barcodes_dev_locked(gtgpu_index* ix, uint64_t n, const uint32_t* d_chr, const uint32_t* d_start,
                                         const uint32_t* d_end, const uint32_t* d_bc, uint32_t n_barcodes,
                                         uint64_t* out_barcode_offsets, gtgpu_buf** out_peaks, gtgpu_buf** out_counts) {
    gtgpu_ctx* ctx = ix->ctx;
    cudaStream_t st = ctx->stream;
    uint64_t nnz = 0, total = 0;
    uint32_t *d_peak_out = nullptr, *d_count_out = nullptr;
    if (n) {
        uint64_t* d_off;
        GT_TRY(ctx->scratch_get(SC_OUT_OFFS, (n + 1) * 8, (void**)&d_off));
        uint32_t* d_ids = nullptr;
        GT_TRY(fused_find_all(ix, n, 0, nullptr, d_chr, d_start, d_end, d_off, nullptr, &d_ids, &total));
        if (total >= 0xFFFFFFFFull) return fail(GTGPU_ERR_UNSUPPORTED, "score_barcodes: more than 2^32-2 hits per call");
        if (total) {
            uint32_t *d_hbc, *d_k2, *d_v2;
            unsigned long long *d_head, *d_rank, *d_runs;
            void* d_tmp;
            uint64_t* d_bco;
            GT_TRY(ctx->scratch_get(SC_IN2_CHR, total * 4, (void**)&d_hbc));
            GT_TRY(ctx->scratch_get(SC_IN2_START, total * 4, (void**)&d_k2));
            GT_TRY(ctx->scratch_get(SC_IN2_END, total * 4, (void**)&d_v2));
            GT_TRY(ctx->scratch_get(SC_IN3_START, std::max(radix_sort_temp_bytes(total), exclusive_scan_temp_bytes(total, 8)), &d_tmp));
            score_hit_barcodes_kernel<<<grid_for(ctx, n), 256, 0, st>>>(n, d_off, d_bc, d_hbc);
            ctx->launches++;
            // stable LSD: by peak first, then by barcode -> sorted by (barcode, peak)
            uint32_t *ka = d_ids, *va = d_hbc, *kb = d_k2, *vb = d_v2;
            int in_b = 0;
            GT_TRY(radix_sort_pairs(ctx, total, ka, va, kb, vb, bits_for((uint64_t)ix->max_val + 1), d_tmp, &in_b));
            if (in_b) { std::swap(ka, kb); std::swap(va, vb); }
            // now (ka = peaks sorted, va = barcodes); second sort keys = barcodes, values = peaks
            GT_TRY(radix_sort_pairs(ctx, total, va, ka, vb, kb, bits_for(n_barcodes), d_tmp, &in_b));
            uint32_t* s_bc = in_b ? vb : va;
            uint32_t* s_pk = in_b ? kb : ka;
            GT_TRY(ctx->scratch_get(SC_COUNTS, total * 8, (void**)&d_head));
            GT_TRY(ctx->scratch_get(SC_IN3_CHR, total * 8, (void**)&d_rank));
            GT_TRY(ctx->scratch_get(SC_IN3_END, total * 8, (void**)&d_runs));
            const int g = grid_for(ctx, total);
            score_run_heads_kernel<<<g, 256, 0, st>>>(total, s_bc, s_pk, d_head);
            ctx->launches++;
            GT_TRY(exclusive_scan<unsigned long long>(ctx, d_head, d_rank, total, d_tmp));
            score_run_starts_kernel<<<g, 256, 0, st>>>(total, d_head, d_rank, d_runs);
            ctx->launches++;
            unsigned long long last[2];
            GT_CUDA(cudaMemcpyAsync(&last[0], d_rank + total - 1, 8, cudaMemcpyDeviceToHost, st));
            GT_CUDA(cudaMemcpyAsync(&last[1], d_head + total - 1, 8, cudaMemcpyDeviceToHost, st));
            GT_CUDA(cudaStreamSynchronize(st));
            nnz = last[0] + last[1];
            GT_TRY(ctx->scratch_get(SC_OUT_IDS2, nnz * 8, (void**)&d_peak_out));
            d_count_out = d_peak_out + nnz;
            score_runs_out_kernel<<<grid_for(ctx, nnz), 256, 0, st>>>(nnz, total, d_runs, s_pk, d_peak_out, d_count_out);
            GT_TRY(ctx->scratch_get(SC_FILE_TOK, ((uint64_t)n_barcodes + 1) * 8, (void**)&d_bco));
            score_barcode_offsets_kernel<<<(n_barcodes + 1 + 255) / 256, 256, 0, st>>>(n_barcodes, nnz, d_runs, s_bc, d_bco);
            ctx->launches += 2;
            GT_CUDA(cudaMemcpyAsync(out_barcode_offsets, d_bco, ((uint64_t)n_barcodes + 1) * 8, cudaMemcpyDeviceToHost, st));
            GT_CUDA(cudaGetLastError());
        }
    }
    if (nnz == 0)
        for (uint32_t b = 0; b <= n_barcodes; ++b) out_barcode_offsets[b] = 0;

    BufPtr peaks, counts;
    int32_t s = buf_from_device(ctx, d_peak_out, nnz, 4, st, &peaks);
    if (s == GTGPU_OK) s = buf_from_device(ctx, d_count_out, nnz, 4, st, &counts);
    if (s != GTGPU_OK) {
        cudaStreamSynchronize(st);  // the peaks' copy may still run
        return s == GTGPU_ERR_CUDA ? fail(s, std::string("score_barcodes: D2H: ") + gtgpu_last_error()) : s;
    }
    const cudaError_t e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) return fail(GTGPU_ERR_CUDA, std::string("score_barcodes: ") + cudaGetErrorString(e));
    *out_peaks = peaks.release();
    *out_counts = counts.release();
    return GTGPU_OK;
}

extern "C" int32_t gtgpu_score_barcodes(gtgpu_index* ix, uint64_t n, const uint32_t* chr, const uint32_t* start,
                                        const uint32_t* end, const uint32_t* barcode_id, uint32_t n_barcodes,
                                        uint64_t* out_barcode_offsets, gtgpu_buf** out_peaks, gtgpu_buf** out_counts) try {
    if (!ix || !out_barcode_offsets || !out_peaks || !out_counts || (n && (!chr || !start || !end || !barcode_id)))
        return fail(GTGPU_ERR_INVALID, "score_barcodes: null argument");
    if (n >= 0xFFFFFFFFull) return fail(GTGPU_ERR_UNSUPPORTED, "score_barcodes: more than 2^32-2 fragments per call");
    for (uint64_t i = 0; i < n; ++i)
        if (barcode_id[i] >= n_barcodes) return fail(GTGPU_ERR_INVALID, "score_barcodes: barcode id out of range");
    gtgpu_ctx* ctx = ix->ctx;
    std::lock_guard<std::mutex> lk(ctx->mu);
    GT_CUDA(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    uint32_t *d_chr = nullptr, *d_start = nullptr, *d_end = nullptr, *d_bc = nullptr;
    if (n) {
        GT_TRY(ctx->scratch_get(SC_CHR, n * 4, (void**)&d_chr));
        GT_TRY(ctx->scratch_get(SC_START, n * 4, (void**)&d_start));
        GT_TRY(ctx->scratch_get(SC_END, n * 4, (void**)&d_end));
        GT_TRY(ctx->scratch_get(SC_BARCODE, n * 4, (void**)&d_bc));
        GT_CUDA(cudaMemcpyAsync(d_chr, chr, n * 4, cudaMemcpyHostToDevice, st));
        GT_CUDA(cudaMemcpyAsync(d_start, start, n * 4, cudaMemcpyHostToDevice, st));
        GT_CUDA(cudaMemcpyAsync(d_end, end, n * 4, cudaMemcpyHostToDevice, st));
        GT_CUDA(cudaMemcpyAsync(d_bc, barcode_id, n * 4, cudaMemcpyHostToDevice, st));
    }
    return score_barcodes_dev_locked(ix, n, d_chr, d_start, d_end, d_bc, n_barcodes, out_barcode_offsets, out_peaks, out_counts);
} GT_CATCH

// ---- region / barcode scoring from a fragment file's bytes -----------------------------------------------------------------
// Each file is parsed in windows (for_each_window, ingest.cu); gzip members are inflated whole into device memory first.
namespace gtgpu {

static int32_t parse_error(const std::string& who, uint64_t line) {
    return fail(GTGPU_ERR_INVALID, who + ": Failed to parse fragment at line " + std::to_string(line));
}

static int32_t too_many(const std::string& who) {
    return fail(GTGPU_ERR_UNSUPPORTED, who + ": more than 2^32 - 1 fragments in one file");
}

// the caller holds ctx->mu
static int32_t score_matrix_text_locked(gtgpu_index* ix, const char* host_text, const char* dev_text, uint64_t n_bytes,
                                        uint32_t n_names, const char* names, const uint32_t* name_offsets, int32_t mode,
                                        uint64_t n_cols, uint32_t* out_row, const std::string& who) {
    gtgpu_ctx* ctx = ix->ctx;
    cudaStream_t st = ctx->stream;
    uint32_t* d_row;
    GT_TRY(ctx->scratch_get(SC_MATRIX, std::max<uint64_t>(n_cols * 4, 4), (void**)&d_row));
    GT_CUDA(cudaMemsetAsync(d_row, 0, n_cols * 4, st));
    if (n_bytes) {
        NameTable nt;
        uint64_t* d_fo;
        uint64_t total = 0;
        GT_TRY(upload_name_table(ctx, n_names, names, name_offsets, &nt));
        GT_TRY(ctx->scratch_get(SC_FILE_OFFS, 16, (void**)&d_fo));
        GT_TRY(for_each_window(ctx, host_text, dev_text, n_bytes, who,
                               [&](const char* d, uint64_t nb, uint64_t, uint64_t line0, uint32_t* n_lines) -> int32_t {
            ParsedLines fp;
            GT_TRY(parse_lines_locked(ctx, d, nb, FRAG_SCORE_MATRIX, nt, BedFilesView{}, &fp));
            *n_lines = fp.n_lines;
            if (fp.bad_line != 0xFFFFFFFFu) return parse_error(who, line0 + fp.bad_line);
            total += fp.n;
            if (total > 0xFFFFFFFFull) return too_many(who);
            const uint64_t fo[2] = {0, fp.n};
            GT_CUDA(cudaMemcpyAsync(d_fo, fo, 16, cudaMemcpyHostToDevice, st));
            GT_TRY(score_matrix_dev_locked(ix, 1, d_fo, fp.n, fp.chr, fp.start, fp.end, mode, n_cols, d_row, true));
            GT_CUDA(cudaStreamSynchronize(st));  // the window's buffers are reused by the next one
            return GTGPU_OK;
        }));
    }
    if (n_cols) GT_CUDA(cudaMemcpyAsync(out_row, d_row, n_cols * 4, cudaMemcpyDeviceToHost, st));
    GT_CUDA(cudaStreamSynchronize(st));
    return GTGPU_OK;
}

// the caller holds ctx->mu
static int32_t score_barcodes_text_locked(gtgpu_index* ix, const char* host_text, const char* dev_text, uint64_t n_bytes,
                                          uint32_t n_names, const char* names, const uint32_t* name_offsets, uint32_t* out_n_barcodes,
                                          gtgpu_buf** out_names, gtgpu_buf** out_name_offsets, gtgpu_buf** out_barcode_offsets,
                                          gtgpu_buf** out_peaks, gtgpu_buf** out_counts, const std::string& who) {
    gtgpu_ctx* ctx = ix->ctx;
    KeyTable tab(false, false, ~0ull, who, "gtgpu_score_barcodes", "barcode", "barcodes");
    if (n_bytes) {
        NameTable nt;
        GT_TRY(upload_name_table(ctx, n_names, names, name_offsets, &nt));
        GT_TRY(for_each_window(ctx, host_text, dev_text, n_bytes, who,
                               [&](const char* d, uint64_t nb, uint64_t byte0, uint64_t line0, uint32_t* n_lines) -> int32_t {
            ParsedLines fp;
            GT_TRY(parse_lines_locked(ctx, d, nb, FRAG_SCORE_BARCODES, nt, BedFilesView{}, &fp));
            *n_lines = fp.n_lines;
            if (fp.bad_line != 0xFFFFFFFFu) return parse_error(who, line0 + fp.bad_line);
            if (tab.n + fp.n > 0xFFFFFFFFull) return too_many(who);
            return tab.add_window(ctx, d, byte0, fp, n_names);
        }));
    }
    uint32_t n_kept = 0;
    BufPtr nm, no, offs;
    GT_TRY(tab.finish(ctx, &n_kept, &nm, &no));
    GT_TRY(buf_new(ctx, (uint64_t)n_kept + 1, 8, &offs));
    GT_TRY(score_barcodes_dev_locked(ix, tab.n, tab.chr.u32(), tab.start.u32(), tab.end.u32(), tab.id.u32(), n_kept,
                                     (uint64_t*)offs->block.ptr, out_peaks, out_counts));
    *out_n_barcodes = n_kept;
    *out_names = nm.release();
    *out_name_offsets = no.release();
    *out_barcode_offsets = offs.release();
    return GTGPU_OK;
}

}  // namespace gtgpu

extern "C" int32_t gtgpu_score_matrix_text(gtgpu_index* ix, const char* text, uint64_t n_bytes, uint32_t n_names, const char* names,
                                           const uint32_t* name_offsets, int32_t mode, uint64_t n_cols, uint32_t* out_row) try {
    if (!ix || (n_cols && !out_row) || (n_bytes && !text) || (n_names && (!names || !name_offsets)))
        return fail(GTGPU_ERR_INVALID, "score_matrix_text: null argument");
    if (mode != GTGPU_SCORE_ATAC && mode != GTGPU_SCORE_CHIP) return fail(GTGPU_ERR_INVALID, "score_matrix_text: unknown mode");
    gtgpu_ctx* ctx = ix->ctx;
    std::lock_guard<std::mutex> lk(ctx->mu);
    GT_CUDA(cudaSetDevice(ctx->device));
    return score_matrix_text_locked(ix, text, nullptr, n_bytes, n_names, names, name_offsets, mode, n_cols, out_row, "score_matrix_text");
} GT_CATCH

extern "C" int32_t gtgpu_score_matrix_gz(gtgpu_index* ix, uint64_t n_members, const uint8_t* gz, const uint64_t* member_offsets,
                                         uint32_t n_names, const char* names, const uint32_t* name_offsets, int32_t mode, uint64_t n_cols,
                                         uint32_t* out_row) try {
    if (!ix || (n_cols && !out_row) || (n_names && (!names || !name_offsets))) return fail(GTGPU_ERR_INVALID, "score_matrix_gz: null argument");
    if (mode != GTGPU_SCORE_ATAC && mode != GTGPU_SCORE_CHIP) return fail(GTGPU_ERR_INVALID, "score_matrix_gz: unknown mode");
    GT_TRY(check_members(n_members, gz, member_offsets, "score_matrix_gz"));
    gtgpu_ctx* ctx = ix->ctx;
    std::lock_guard<std::mutex> lk(ctx->mu);
    GT_CUDA(cudaSetDevice(ctx->device));
    uint8_t* d_text = nullptr;
    uint64_t n_text = 0;
    GT_TRY(inflate_whole_locked(ctx, n_members, gz, member_offsets, "score_matrix_gz", &d_text, &n_text));
    return score_matrix_text_locked(ix, nullptr, (const char*)d_text, n_text, n_names, names, name_offsets, mode, n_cols, out_row,
                                    "score_matrix_gz");
} GT_CATCH

extern "C" int32_t gtgpu_score_barcodes_text(gtgpu_index* ix, const char* text, uint64_t n_bytes, uint32_t n_names, const char* names,
                                             const uint32_t* name_offsets, uint32_t* out_n_barcodes, gtgpu_buf** out_barcode_names,
                                             gtgpu_buf** out_barcode_name_offsets, gtgpu_buf** out_barcode_offsets,
                                             gtgpu_buf** out_peaks, gtgpu_buf** out_counts) try {
    if (!ix || !out_n_barcodes || !out_barcode_names || !out_barcode_name_offsets || !out_barcode_offsets || !out_peaks || !out_counts ||
        (n_bytes && !text) || (n_names && (!names || !name_offsets)))
        return fail(GTGPU_ERR_INVALID, "score_barcodes_text: null argument");
    gtgpu_ctx* ctx = ix->ctx;
    std::lock_guard<std::mutex> lk(ctx->mu);
    GT_CUDA(cudaSetDevice(ctx->device));
    return score_barcodes_text_locked(ix, text, nullptr, n_bytes, n_names, names, name_offsets, out_n_barcodes, out_barcode_names,
                                      out_barcode_name_offsets, out_barcode_offsets, out_peaks, out_counts, "score_barcodes_text");
} GT_CATCH

extern "C" int32_t gtgpu_score_barcodes_gz(gtgpu_index* ix, uint64_t n_members, const uint8_t* gz, const uint64_t* member_offsets,
                                           uint32_t n_names, const char* names, const uint32_t* name_offsets, uint32_t* out_n_barcodes,
                                           gtgpu_buf** out_barcode_names, gtgpu_buf** out_barcode_name_offsets,
                                           gtgpu_buf** out_barcode_offsets, gtgpu_buf** out_peaks, gtgpu_buf** out_counts) try {
    if (!ix || !out_n_barcodes || !out_barcode_names || !out_barcode_name_offsets || !out_barcode_offsets || !out_peaks || !out_counts ||
        (n_names && (!names || !name_offsets)))
        return fail(GTGPU_ERR_INVALID, "score_barcodes_gz: null argument");
    GT_TRY(check_members(n_members, gz, member_offsets, "score_barcodes_gz"));
    gtgpu_ctx* ctx = ix->ctx;
    std::lock_guard<std::mutex> lk(ctx->mu);
    GT_CUDA(cudaSetDevice(ctx->device));
    uint8_t* d_text = nullptr;
    uint64_t n_text = 0;
    GT_TRY(inflate_whole_locked(ctx, n_members, gz, member_offsets, "score_barcodes_gz", &d_text, &n_text));
    return score_barcodes_text_locked(ix, nullptr, (const char*)d_text, n_text, n_names, names, name_offsets, out_n_barcodes,
                                      out_barcode_names, out_barcode_name_offsets, out_barcode_offsets, out_peaks, out_counts,
                                      "score_barcodes_gz");
} GT_CATCH
