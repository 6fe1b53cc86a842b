// sort_shim.cpp — test-only C entry points to the device primitives of sort.cu, which are not part of the C ABI.
//
// The prototypes below are copied from gtars_b200/csrc/cuda/common.cuh and resolve against libgtars_gpu.so (built with
// default visibility; the two exclusive_scan instantiations are weak symbols of sort.cu).  When a prototype there changes,
// this file stops linking and has to change with it.  tests/test_gpu_sort.py builds it with g++ into a temporary directory.
#include <cstddef>
#include <cstdint>

struct gtgpu_ctx;

namespace gtgpu {
size_t exclusive_scan_temp_bytes(uint64_t n, size_t elem);
template <typename T>
int32_t exclusive_scan(gtgpu_ctx* ctx, const T* d_in, T* d_out, uint64_t n, void* d_temp);
int32_t inclusive_max_scan_u64(gtgpu_ctx* ctx, const unsigned long long* d_in, unsigned long long* d_out, uint64_t n, void* d_temp);
size_t radix_sort_temp_bytes(uint64_t n);
int32_t radix_sort_pairs(gtgpu_ctx* ctx, uint64_t n, uint32_t* keys_a, uint32_t* vals_a, uint32_t* keys_b, uint32_t* vals_b,
                         int bits, void* d_temp, int* result_in_b, const uint64_t* d_n);
void radix_plan(int bits, int* passes, int* width);
bool radix_group_fits(uint32_t n_keys, uint32_t max_val);
size_t radix_group_temp_bytes(uint64_t n, uint32_t n_keys);
int32_t radix_group_values(gtgpu_ctx* ctx, uint64_t n_cap, const uint32_t* keys, const uint32_t* vals, uint32_t* packed_tmp,
                           uint32_t* vals_out, uint32_t n_keys, uint32_t max_val, void* d_temp, const uint64_t* d_n,
                           uint64_t* out_offsets, uint64_t* d_total);
}  // namespace gtgpu

extern "C" {
size_t shim_exclusive_scan_temp_bytes(uint64_t n, size_t elem) { return gtgpu::exclusive_scan_temp_bytes(n, elem); }
int32_t shim_exclusive_scan_u32(gtgpu_ctx* ctx, const uint32_t* in, uint32_t* out, uint64_t n, void* tmp) {
    return gtgpu::exclusive_scan<uint32_t>(ctx, in, out, n, tmp);
}
int32_t shim_exclusive_scan_u64(gtgpu_ctx* ctx, const unsigned long long* in, unsigned long long* out, uint64_t n, void* tmp) {
    return gtgpu::exclusive_scan<unsigned long long>(ctx, in, out, n, tmp);
}
int32_t shim_inclusive_max_scan_u64(gtgpu_ctx* ctx, const unsigned long long* in, unsigned long long* out, uint64_t n, void* tmp) {
    return gtgpu::inclusive_max_scan_u64(ctx, in, out, n, tmp);
}
size_t shim_radix_sort_temp_bytes(uint64_t n) { return gtgpu::radix_sort_temp_bytes(n); }
int32_t shim_radix_sort_pairs(gtgpu_ctx* ctx, uint64_t n, uint32_t* keys_a, uint32_t* vals_a, uint32_t* keys_b, uint32_t* vals_b,
                              int bits, void* tmp, int* result_in_b, const uint64_t* d_n) {
    return gtgpu::radix_sort_pairs(ctx, n, keys_a, vals_a, keys_b, vals_b, bits, tmp, result_in_b, d_n);
}
void shim_radix_plan(int bits, int* passes, int* width) { gtgpu::radix_plan(bits, passes, width); }
int32_t shim_radix_group_fits(uint32_t n_keys, uint32_t max_val) { return gtgpu::radix_group_fits(n_keys, max_val) ? 1 : 0; }
size_t shim_radix_group_temp_bytes(uint64_t n, uint32_t n_keys) { return gtgpu::radix_group_temp_bytes(n, n_keys); }
int32_t shim_radix_group_values(gtgpu_ctx* ctx, uint64_t n_cap, const uint32_t* keys, const uint32_t* vals, uint32_t* packed_tmp,
                                uint32_t* vals_out, uint32_t n_keys, uint32_t max_val, void* tmp, const uint64_t* d_n,
                                uint64_t* out_offsets, uint64_t* d_total) {
    return gtgpu::radix_group_values(ctx, n_cap, keys, vals, packed_tmp, vals_out, n_keys, max_val, tmp, d_n, out_offsets, d_total);
}
}
