// fragments.cu — tokenize_fragment_file on the device (gtars-tokenizers/src/utils/fragments.rs:12-82).
//
// Every fragment is its own Tokenizer::tokenize call, so a fragment without a hit (or on an unknown chromosome)
// contributes one unk id; ids are appended to the fragment's barcode list in input order.  Device plan:
//   1. fused find over all fragments with the per-query [unk] rule and per-fragment offsets (kernels.cu): its id stream
//      IS the token stream in fragment order, a fragment's tokens are [off[i], off[i+1])
//   2. every token gets its fragment's barcode as a tag (one coalesced pass)
//   3. stable LSD radix sort of (barcode, token) pairs by barcode (sort.cu, hand-written; 2 passes of 9 bits for 100 k
//      barcodes): the sorted tokens are the output, barcode-major, input order kept inside a barcode
//   4. barcode offsets by binary search over the sorted tags
//   3+4 for barcodes of 10-18 bits whose upper digit fits next to a token in 32 bits (the usual case): radix_group_values —
//      pass 1 writes packed (upper digit | token) words, pass 2 sorts those and writes bare tokens, offsets from counts
// Nothing is gathered at random: every pass streams (the first version sorted fragment indices and then chased offsets
// and ids per fragment — 190 ms per 1e9 fragments, against ~45 ms for this one).
// Output is barcode-major: out_barcode_offsets[n_barcodes + 1] + ids.
#include <algorithm>
#include <cstring>

#include "common.cuh"

namespace gtgpu {

// tag[j] = barcode of the fragment that token j belongs to; four fragments per thread keep the offset loads wide
// run_if (optional): the find wrote the tags itself unless this device flag is non-zero (its lean kernel fell back)
__global__ void frag_tag_tokens_kernel(uint64_t n, const uint64_t* __restrict__ offsets, const uint32_t* __restrict__ barcode,
                                       uint64_t capacity, uint32_t* __restrict__ tags, const uint32_t* __restrict__ run_if) {
    if (run_if && *run_if == 0) return;
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        const uint64_t a = offsets[i], b = min(offsets[i + 1], capacity);
        const uint32_t bc = barcode[i];
        for (uint64_t j = a; j < b; ++j) tags[j] = bc;
    }
}

// out[b] = first position of the sorted tags holding a barcode >= b, for b in [0, n_barcodes]; *d_total = number of tokens
// (or ~0 when the find produced more tokens than the buffers hold: the result is then incomplete)
__global__ void frag_barcode_offsets_kernel(uint32_t n_barcodes, const uint64_t* __restrict__ d_n, uint64_t capacity,
                                            const uint32_t* __restrict__ sorted_tags, uint64_t* __restrict__ out,
                                            uint64_t* __restrict__ d_total) {
    const uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b > n_barcodes) return;
    const uint64_t n = min((uint64_t)*d_n, capacity);
    uint64_t lo = 0, hi = n;
    while (lo < hi) {
        const uint64_t mid = (lo + hi) >> 1;
        if (sorted_tags[mid] < b) lo = mid + 1;
        else hi = mid;
    }
    out[b] = lo;
    if (b == 0 && d_total) *d_total = *d_n > capacity ? ~0ull : *d_n;
}

// Steps 1-4 on device-resident fragments, queued on the ctx stream without a host synchronisation.  The tokens land in
// d_out (capacity cap ids); d_alt / d_tag_a / d_tag_b are scratch of the same capacity.  The caller holds ctx->mu.
// d_ntok (device) receives the number of tokens the find produced (may exceed cap: the caller checks).
static int32_t fragments_group_by(gtgpu_index* ix, uint64_t n, const uint32_t* d_chr, const uint32_t* d_start, const uint32_t* d_end,
                                  const uint32_t* d_bc, uint32_t n_barcodes, uint32_t unk_id, uint64_t cap, uint32_t* d_out,
                                  uint32_t* d_alt, uint32_t* d_tag_a, uint32_t* d_tag_b, uint64_t* d_off, void* d_ws, void* d_sort_tmp,
                                  uint64_t* d_misc, uint64_t* d_bco, uint64_t* d_total_or_null, int stage, const uint32_t** tag_if) {
    gtgpu_ctx* ctx = ix->ctx;
    cudaStream_t st = ctx->stream;
    int bits = 1;
    while (bits < 32 && (1ull << bits) < n_barcodes) ++bits;
    int passes, width;
    radix_plan(bits, &passes, &width);
    // the sort ping-pongs between two buffers: start in the one that makes the LAST pass write into d_out
    uint32_t* first = (passes & 1) ? d_alt : d_out;
    uint32_t* second = (passes & 1) ? d_out : d_alt;
    if (stage == 0 || stage == 1) {
        GT_CUDA(cudaMemsetAsync(d_misc, 0, 64, st));
        // the find writes (token, barcode) pairs itself when its lean kernel serves the index; *tag_if then is the device
        // flag of the exception (fallback to the full kernel: offsets were written, step 2 tags from them)
        GT_TRY(launch_fused_find(ix, n, 0, nullptr, d_chr, d_start, d_end, 0, first, cap, d_off, nullptr, d_ws, nullptr, d_misc,
                                 (uint32_t*)(d_misc + 2), 1, unk_id, d_bc, d_tag_a, tag_if));
    }
    if (stage == 0 || stage == 2) {
        const int grid = (int)std::min<uint64_t>((n + 255) / 256, (uint64_t)ctx->sm_count * 16);
        frag_tag_tokens_kernel<<<grid, 256, 0, st>>>(n, d_off, d_bc, cap, d_tag_a, *tag_if);
        ctx->launches++;
        const uint32_t max_token = std::max(ix->max_val, unk_id);
        if (radix_group_fits(n_barcodes, max_token)) {
            // two digit passes and the barcode's upper digit fits next to a token: the second pass sorts packed words and the
            // barcode offsets come from counts (sort.cu, radix_group_values) — no sorted tags, 20 instead of 32 B per token
            GT_TRY(radix_group_values(ctx, cap, d_tag_a, first, d_tag_b, d_out, n_barcodes, max_token, d_sort_tmp, d_misc, d_bco,
                                      d_total_or_null));
        } else {
            int in_b = 0;
            GT_TRY(radix_sort_pairs(ctx, cap, d_tag_a, first, d_tag_b, second, bits, d_sort_tmp, &in_b, d_misc));
            const uint32_t* sorted_tags = in_b ? d_tag_b : d_tag_a;
            frag_barcode_offsets_kernel<<<(n_barcodes + 1 + 255) / 256, 256, 0, st>>>(n_barcodes, d_misc, cap, sorted_tags, d_bco, d_total_or_null);
            ctx->launches++;
        }
        GT_CUDA(cudaGetLastError());
    }
    return GTGPU_OK;
}

}  // namespace gtgpu

using namespace gtgpu;

namespace gtgpu {

// Device-resident core (the caller holds ctx->mu): fragments in d_chr / d_start / d_end, dense barcode ids in d_bc.
int32_t tokenize_fragments_core(gtgpu_index* ix, uint64_t n, const uint32_t* d_chr, const uint32_t* d_start, const uint32_t* d_end,
                                uint32_t* d_bc, uint32_t n_barcodes, uint32_t unk_id, uint64_t* out_barcode_offsets, BufPtr* out_ids) {
    gtgpu_ctx* ctx = ix->ctx;
    cudaStream_t st = ctx->stream;
    if (n == 0) {
        for (uint32_t b = 0; b <= n_barcodes; ++b) out_barcode_offsets[b] = 0;
        return buf_new(ctx, 0, 4, out_ids);
    }
    uint32_t *d_out = nullptr, *d_alt = nullptr, *d_tag_a = nullptr, *d_tag_b = nullptr;
    uint64_t *d_off, *d_bco, *d_misc;
    void *d_ws, *d_tmp;
    GT_TRY(ctx->scratch_get(SC_OUT_OFFS, (n + 1) * 8, (void**)&d_off));
    GT_TRY(ctx->scratch_get(SC_FILE_TOK, ((uint64_t)n_barcodes + 1) * 8, (void**)&d_bco));
    GT_TRY(ctx->scratch_get(SC_TILE_STATUS, fused_workspace_bytes(n), &d_ws));
    GT_TRY(ctx->scratch_get(SC_MISC, 64, (void**)&d_misc));
    uint64_t cap = n + n / 4 + 1024, total = 0;
    const uint32_t* tag_if = nullptr;  // set by step 1, read by step 2
    for (int attempt = 0; attempt < 2; ++attempt) {
        if (cap >= 0xFFFFFFFFull) return fail(GTGPU_ERR_UNSUPPORTED, "tokenize_fragments: more than 2^32-2 tokens per call");
        GT_TRY(ctx->scratch_get(SC_OUT_IDS, cap * 4, (void**)&d_out));
        GT_TRY(ctx->scratch_get(SC_OUT_IDS2, cap * 4, (void**)&d_alt));
        GT_TRY(ctx->scratch_get(SC_IN2_CHR, cap * 4, (void**)&d_tag_a));
        GT_TRY(ctx->scratch_get(SC_IN2_START, cap * 4, (void**)&d_tag_b));
        GT_TRY(ctx->scratch_get(SC_IN3_START, radix_group_temp_bytes(cap, n_barcodes), &d_tmp));
        // 1. tokens of every fragment in fragment order (hits, or unk), with per-fragment offsets
        GT_TRY(fragments_group_by(ix, n, d_chr, d_start, d_end, d_bc, n_barcodes, unk_id, cap, d_out, d_alt, d_tag_a, d_tag_b, d_off,
                                  d_ws, d_tmp, d_misc, d_bco, nullptr, 1, &tag_if));
        GT_CUDA(cudaMemcpyAsync(ctx->h_scalars, d_misc, 24, cudaMemcpyDeviceToHost, st));
        GT_CUDA(cudaStreamSynchronize(st));
        total = ctx->h_scalars[0];
        if ((uint32_t)ctx->h_scalars[2] != 0) return fail(GTGPU_ERR_UNSUPPORTED, "tokenize_fragments: tile overflow");
        if (total <= cap) break;
        if (attempt == 1) return fail(GTGPU_ERR_CAPACITY, "tokenize_fragments: output capacity exceeded twice");
        cap = total;  // multi-hit universes: redo with an exact buffer
    }
    // 2.-4. tag, sort by barcode, offsets
    GT_TRY(fragments_group_by(ix, n, d_chr, d_start, d_end, d_bc, n_barcodes, unk_id, cap, d_out, d_alt, d_tag_a, d_tag_b, d_off, d_ws,
                              d_tmp, d_misc, d_bco, nullptr, 2, &tag_if));
    GT_CUDA(cudaMemcpyAsync(out_barcode_offsets, d_bco, ((uint64_t)n_barcodes + 1) * 8, cudaMemcpyDeviceToHost, st));

    BufPtr buf;
    const int32_t s = buf_from_device(ctx, d_out, total, 4, st, &buf);
    if (s == GTGPU_ERR_CUDA) return fail(s, std::string("tokenize_fragments: D2H: ") + gtgpu_last_error());
    GT_TRY(s);
    const cudaError_t e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) return fail(GTGPU_ERR_CUDA, std::string("tokenize_fragments: D2H: ") + cudaGetErrorString(e));
    *out_ids = std::move(buf);
    return GTGPU_OK;
}

}  // namespace gtgpu

static int32_t tokenize_fragments_one(gtgpu_index* ix, uint64_t n, const uint32_t* chr, const uint32_t* start, const uint32_t* end,
                                      const uint32_t* barcode_id, uint32_t n_barcodes, uint32_t unk_id,
                                      uint64_t* out_barcode_offsets, BufPtr* out_ids) {
    gtgpu_ctx* ctx = ix->ctx;
    std::lock_guard<std::mutex> lk(ctx->mu);
    GT_CUDA(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    uint32_t *d_chr, *d_start, *d_end, *d_bc;
    GT_TRY(ctx->scratch_get(SC_CHR, n * 4, (void**)&d_chr));
    GT_TRY(ctx->scratch_get(SC_START, n * 4, (void**)&d_start));
    GT_TRY(ctx->scratch_get(SC_END, n * 4, (void**)&d_end));
    GT_TRY(ctx->scratch_get(SC_BARCODE, n * 4, (void**)&d_bc));
    if (n) {
        GT_CUDA(cudaMemcpyAsync(d_chr, chr, n * 4, cudaMemcpyHostToDevice, st));
        GT_CUDA(cudaMemcpyAsync(d_start, start, n * 4, cudaMemcpyHostToDevice, st));
        GT_CUDA(cudaMemcpyAsync(d_end, end, n * 4, cudaMemcpyHostToDevice, st));
        GT_CUDA(cudaMemcpyAsync(d_bc, barcode_id, n * 4, cudaMemcpyHostToDevice, st));
    }
    return tokenize_fragments_core(ix, n, d_chr, d_start, d_end, d_bc, n_barcodes, unk_id, out_barcode_offsets, out_ids);
}

// Multi-device group: the fragments are dealt to the devices in contiguous blocks, every device groups its block by
// barcode, and each barcode's final list is the concatenation of its per-device lists in device order — file order inside
// a barcode is preserved because the blocks are contiguous ranges of the file (SURVEY 8e; no collective).
static int32_t tokenize_fragments_group(gtgpu_index* ix, uint64_t n, const uint32_t* chr, const uint32_t* start, const uint32_t* end,
                                        const uint32_t* barcode_id, uint32_t n_barcodes, uint32_t unk_id,
                                        uint64_t* out_barcode_offsets, gtgpu_buf** out_ids) {
    std::lock_guard<std::mutex> glk(ix->ctx->group_mu);
    const size_t D = ix->replicas.size();
    std::vector<BufPtr> parts(D);
    std::vector<std::vector<uint64_t>> offs(D, std::vector<uint64_t>((size_t)n_barcodes + 1, 0));
    int32_t s = for_each_device(D, [&](size_t r) -> int32_t {
        uint64_t lo, hi;
        block_range(n, D, r, &lo, &hi);
        return tokenize_fragments_one(ix->replicas[r], hi - lo, chr + lo, start + lo, end + lo, barcode_id + lo, n_barcodes, unk_id,
                                      offs[r].data(), &parts[r]);
    });
    BufPtr buf;
    if (s == GTGPU_OK) {
        out_barcode_offsets[0] = 0;
        for (uint32_t b = 0; b < n_barcodes; ++b) {
            uint64_t len = 0;
            for (size_t r = 0; r < D; ++r) len += offs[r][b + 1] - offs[r][b];
            out_barcode_offsets[b + 1] = out_barcode_offsets[b] + len;
        }
        cudaSetDevice(ix->ctx->device);
        s = buf_new(ix->ctx, out_barcode_offsets[n_barcodes], 4, &buf);
    }
    if (s == GTGPU_OK) {
        uint32_t* dst = (uint32_t*)buf->block.ptr;
        for_each_device(D, [&](size_t t) -> int32_t {  // D host threads, each a contiguous range of barcodes
            uint64_t b0, b1;
            block_range(n_barcodes, D, t, &b0, &b1);
            for (uint64_t b = b0; b < b1; ++b) {
                uint64_t pos = out_barcode_offsets[b];
                for (size_t r = 0; r < D; ++r) {
                    const uint64_t a = offs[r][b], len = offs[r][b + 1] - a;
                    if (len) memcpy(dst + pos, (const uint32_t*)parts[r]->block.ptr + a, len * 4);
                    pos += len;
                }
            }
            return GTGPU_OK;
        });
        *out_ids = buf.release();
    }
    return s;
}

extern "C" int32_t gtgpu_tokenize_fragments(gtgpu_index* ix, uint64_t n, const uint32_t* chr, const uint32_t* start,
                                            const uint32_t* end, const uint32_t* barcode_id, uint32_t n_barcodes,
                                            uint32_t unk_id, uint64_t* out_barcode_offsets, gtgpu_buf** out_ids) try {
    if (!ix || !out_barcode_offsets || !out_ids || (n && (!chr || !start || !end || !barcode_id)))
        return fail(GTGPU_ERR_INVALID, "tokenize_fragments: null argument");
    if (n >= 0xFFFFFFFFull) return fail(GTGPU_ERR_UNSUPPORTED, "tokenize_fragments: more than 2^32-2 fragments per call");
    for (uint64_t i = 0; i < n; ++i)
        if (barcode_id[i] >= n_barcodes) return fail(GTGPU_ERR_INVALID, "tokenize_fragments: barcode id out of range");
    if (ix->replicas.size() > 1 && n >= (1u << 20))
        return tokenize_fragments_group(ix, n, chr, start, end, barcode_id, n_barcodes, unk_id, out_barcode_offsets, out_ids);
    BufPtr ids;
    GT_TRY(tokenize_fragments_one(ix, n, chr, start, end, barcode_id, n_barcodes, unk_id, out_barcode_offsets, &ids));
    *out_ids = ids.release();
    return GTGPU_OK;
} GT_CATCH

// Device-resident form of gtgpu_tokenize_fragments: nothing crosses PCIe and nothing synchronises — find, tagging, the
// stable radix sort by barcode and the offsets are queued on the ctx stream.
extern "C" int32_t gtgpu_tokenize_fragments_dev(gtgpu_index* ix, uint64_t n, const uint32_t* d_chr, const uint32_t* d_start,
                                                const uint32_t* d_end, const uint32_t* d_barcode_id, uint32_t n_barcodes,
                                                uint32_t unk_id, uint64_t* d_out_barcode_offsets, uint32_t* d_out_ids,
                                                uint64_t ids_capacity, uint64_t* d_out_total) try {
    if (!ix || !d_out_barcode_offsets || !d_out_total || (ids_capacity && !d_out_ids) ||
        (n && (!d_chr || !d_start || !d_end || !d_barcode_id)))
        return fail(GTGPU_ERR_INVALID, "tokenize_fragments_dev: null argument");
    if (n >= 0xFFFFFFFFull || ids_capacity >= 0xFFFFFFFFull)
        return fail(GTGPU_ERR_UNSUPPORTED, "tokenize_fragments_dev: more than 2^32-2 fragments / ids per call");
    gtgpu_ctx* ctx = ix->ctx;
    std::lock_guard<std::mutex> lk(ctx->mu);
    GT_CUDA(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    if (n == 0) {
        GT_CUDA(cudaMemsetAsync(d_out_barcode_offsets, 0, ((uint64_t)n_barcodes + 1) * 8, st));
        GT_CUDA(cudaMemsetAsync(d_out_total, 0, 8, st));
        return GTGPU_OK;
    }
    if (ids_capacity < n) return fail(GTGPU_ERR_CAPACITY, "tokenize_fragments_dev: every fragment yields at least one id (ids_capacity < n)");
    uint32_t *d_alt, *d_tag_a, *d_tag_b;
    uint64_t *d_off, *d_misc;
    void *d_ws, *d_tmp;
    const uint64_t cap = ids_capacity;
    GT_TRY(ctx->scratch_get(SC_OUT_IDS2, cap * 4, (void**)&d_alt));
    GT_TRY(ctx->scratch_get(SC_IN2_CHR, cap * 4, (void**)&d_tag_a));
    GT_TRY(ctx->scratch_get(SC_IN2_START, cap * 4, (void**)&d_tag_b));
    GT_TRY(ctx->scratch_get(SC_OUT_OFFS, (n + 1) * 8, (void**)&d_off));
    GT_TRY(ctx->scratch_get(SC_TILE_STATUS, fused_workspace_bytes(n), &d_ws));
    GT_TRY(ctx->scratch_get(SC_MISC, 64, (void**)&d_misc));
    GT_TRY(ctx->scratch_get(SC_IN3_START, radix_group_temp_bytes(cap, n_barcodes), &d_tmp));
    const uint32_t* tag_if = nullptr;
    return fragments_group_by(ix, n, d_chr, d_start, d_end, d_barcode_id, n_barcodes, unk_id, cap, d_out_ids, d_alt, d_tag_a, d_tag_b,
                              d_off, d_ws, d_tmp, d_misc, d_out_barcode_offsets, d_out_total, 0, &tag_if);
} GT_CATCH
