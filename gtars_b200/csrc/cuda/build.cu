// build.cu — device-side primitives of the index builders (gtgpu_index_build, gtgpu_igd_build).
//
// The reference builds its indexes with comparison sorts on the host (Bits::build: sort by (start, end), bits.rs:105;
// AIList::build: sort_by_key(start), ailist.rs:111; Igd::finalize: per-tile sort by start, igd.rs:157-167).  Here the
// ordering is a stable LSD radix sort of a PERMUTATION on the device (sort.cu's hand-written radix passes), one key
// array after the other from the least to the most significant one, so ties keep their input order exactly like the
// reference's stable sorts; running maxima come from the 64-bit max-scan and the bin LUTs from one binary search per
// bin.  A 2x10^8-record LOLA database is ordered in well under a second instead of ~90 s of std::stable_sort.
#include <algorithm>

#include "common.cuh"

namespace gtgpu {

__global__ void build_iota_kernel(uint64_t n, uint32_t* __restrict__ out) {
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) out[i] = (uint32_t)i;
}

__global__ void build_gather_u32_kernel(uint64_t n, const uint32_t* __restrict__ src, const uint32_t* __restrict__ perm,
                                        uint32_t* __restrict__ out) {
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) out[i] = __ldg(src + perm[i]);
}

__global__ void build_max_u32_kernel(uint64_t n, const uint32_t* __restrict__ src, uint32_t* __restrict__ out_max) {
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    uint32_t m = 0;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) m = max(m, src[i]);
    m = __reduce_max_sync(0xFFFFFFFFu, m);
    if ((threadIdx.x & 31) == 0 && m) atomicMax(out_max, m);
}

// out[k] = first position of `sorted` (ascending) holding a value >= k, for k in [0, n_keys]
__global__ void build_key_offsets_kernel(uint64_t n, const uint32_t* __restrict__ sorted, uint32_t n_keys,
                                         uint32_t* __restrict__ out) {
    const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k > n_keys) return;
    uint64_t lo = 0, hi = n;
    while (lo < hi) {
        const uint64_t mid = (lo + hi) >> 1;
        if (sorted[mid] < k) lo = mid + 1;
        else hi = mid;
    }
    out[k] = (uint32_t)lo;
}

// One LUT family per descriptor: lut[d.lut_off + b] = lower_bound(arr[d.arr_off .. d.arr_off + d.len), b << shift) for
// b in [0, d.nb], entry nb = len.  Descriptors are laid out back to back; `bin_prefix` (n_desc + 1) counts their
// entries (nb + 1 each), so a flat thread index finds its descriptor with one small binary search.
__global__ void build_luts_kernel(uint32_t n_desc, const LutDesc* __restrict__ desc, const uint64_t* __restrict__ bin_prefix,
                                  const uint32_t* __restrict__ arr, uint32_t shift, uint32_t* __restrict__ lut) {
    const uint64_t total = bin_prefix[n_desc];
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += stride) {
        uint32_t a = 0, z = n_desc;  // last descriptor whose prefix is <= t
        while (z - a > 1) {
            const uint32_t m = (a + z) >> 1;
            if (bin_prefix[m] <= t) a = m;
            else z = m;
        }
        const LutDesc d = desc[a];
        const uint32_t b = (uint32_t)(t - bin_prefix[a]);
        uint32_t r = d.len;
        if (b < d.nb) {
            const uint64_t key = (uint64_t)b << shift;
            uint32_t lo = 0, hi = d.len;
            const uint32_t* p = arr + d.arr_off;
            while (lo < hi) {
                const uint32_t mid = (lo + hi) >> 1;
                if ((uint64_t)__ldg(p + mid) < key) lo = mid + 1;
                else hi = mid;
            }
            r = lo;
        }
        lut[(uint64_t)d.lut_off + b] = r;
    }
}

int32_t launch_build_luts(gtgpu_ctx* ctx, uint32_t n_desc, const LutDesc* d_desc, const uint64_t* d_bin_prefix, uint64_t total_bins,
                          const uint32_t* d_arr, uint32_t shift, uint32_t* d_lut) {
    if (!n_desc || !total_bins) return GTGPU_OK;
    const int grid = (int)std::min<uint64_t>((total_bins + 255) / 256, (uint64_t)ctx->sm_count * 16);
    build_luts_kernel<<<grid, 256, 0, ctx->stream>>>(n_desc, d_desc, d_bin_prefix, d_arr, shift, d_lut);
    ctx->launches++;
    GT_CUDA(cudaGetLastError());
    return GTGPU_OK;
}

int32_t launch_gather_u32(gtgpu_ctx* ctx, uint64_t n, const uint32_t* d_src, const uint32_t* d_perm, uint32_t* d_out) {
    if (!n) return GTGPU_OK;
    build_gather_u32_kernel<<<grid_for(ctx, n), 256, 0, ctx->stream>>>(n, d_src, d_perm, d_out);
    ctx->launches++;
    GT_CUDA(cudaGetLastError());
    return GTGPU_OK;
}

int32_t launch_key_offsets(gtgpu_ctx* ctx, uint64_t n, const uint32_t* d_sorted, uint32_t n_keys, uint32_t* d_out) {
    build_key_offsets_kernel<<<(n_keys + 1 + 255) / 256, 256, 0, ctx->stream>>>(n, d_sorted, n_keys, d_out);
    ctx->launches++;
    GT_CUDA(cudaGetLastError());
    return GTGPU_OK;
}

int bits_for_value(uint64_t max_value) {
    int b = 1;
    while (b < 32 && (max_value >> b) != 0) ++b;
    return b;
}

// ---- PermSorter -------------------------------------------------------------------------------------------------------
int32_t PermSorter::init(gtgpu_ctx* c, uint64_t count) {
    ctx = c;
    n = count;
    const size_t bytes = std::max<size_t>(n * 4, 16);
    for (uint32_t** p : {&perm, &perm_alt, &key, &key_alt}) {
        cudaError_t e = cudaMalloc((void**)p, bytes);
        if (e != cudaSuccess) return fail(GTGPU_ERR_NOMEM, std::string("cudaMalloc(build sort): ") + cudaGetErrorString(e));
    }
    cudaError_t e = cudaMalloc(&tmp, std::max<size_t>(radix_sort_temp_bytes(n), 256));
    if (e != cudaSuccess) return fail(GTGPU_ERR_NOMEM, std::string("cudaMalloc(build sort): ") + cudaGetErrorString(e));
    e = cudaMalloc((void**)&d_max, 16);
    if (e != cudaSuccess) return fail(GTGPU_ERR_NOMEM, std::string("cudaMalloc(build sort): ") + cudaGetErrorString(e));
    if (n) {
        build_iota_kernel<<<grid_for(ctx, n), 256, 0, ctx->stream>>>(n, perm);
        ctx->launches++;
    }
    GT_CUDA(cudaGetLastError());
    return GTGPU_OK;
}

PermSorter::~PermSorter() {
    for (void* p : {(void*)perm, (void*)perm_alt, (void*)key, (void*)key_alt, tmp, (void*)d_max})
        if (p) cudaFree(p);
}

// One key of the composite ordering (call from the least significant key to the most significant one): the current
// permutation is re-sorted, stably, by src[perm[i]].  bits <= 0: the number of significant bits is measured first.
int32_t PermSorter::pass(const uint32_t* d_src, int bits) {
    if (n == 0) return GTGPU_OK;
    GT_TRY(launch_gather_u32(ctx, n, d_src, perm, key));
    if (bits <= 0) {
        uint32_t h_max = 0;
        GT_CUDA(cudaMemsetAsync(d_max, 0, 4, ctx->stream));
        build_max_u32_kernel<<<grid_for(ctx, n), 256, 0, ctx->stream>>>(n, key, d_max);
        ctx->launches++;
        GT_CUDA(cudaMemcpyAsync(&h_max, d_max, 4, cudaMemcpyDeviceToHost, ctx->stream));
        GT_CUDA(cudaStreamSynchronize(ctx->stream));
        bits = bits_for_value(h_max);
    }
    int in_b = 0;
    GT_TRY(radix_sort_pairs(ctx, n, key, perm, key_alt, perm_alt, bits, tmp, &in_b));
    if (in_b) {
        std::swap(key, key_alt);
        std::swap(perm, perm_alt);
    }
    return GTGPU_OK;
}

}  // namespace gtgpu
