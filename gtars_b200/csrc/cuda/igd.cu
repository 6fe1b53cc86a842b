// igd.cu — gtars-igd / gtars-lola overlap-count matrices on the device.
//
// The reference (gtars-igd/src/igd.rs) bins every database interval into 16 384-bp tiles and walks, per query, every
// record of the touched tiles (igd.rs:753-847).  For min_overlap >= 1 the result is tile-independent (SURVEY.md A.5):
//     hit(q, r, m)  <=>  same contig  &&  r.start < q.end  &&  min(r.end, q.end) - max(r.start, max(q.start, 0)) >= m
// so the device keeps, per contig, ONE pooled start-sorted SoA of all database records (start, end, file) plus
//   pmax[i]  = max end over records [0, i]            -> candidate range [first i with pmax > q.start, #starts < q.end)
//   psame[i] = max end over EARLIER records of the same file with length >= m (m = 1 precomputed)
// One warp resolves one query: the lanes stride over the candidate range, test the closed form and add into the
// [n_sets x n_files] matrix with 64-bit atomics (the 80 MB matrix of the LOLA configuration is L2-resident).
//   count_set_overlaps (igd.rs:544-556): every hit counts.
//   count_region_hits  (igd.rs:563-590): a (query, file) pair counts once.  A hit r is the FIRST hit of its file for
//       this query iff no earlier same-file record hits, i.e. iff psame[r] - q.start < m (derivation in DESIGN.md);
//       that replaces the reference's O(n_files) scratch zero + scan per region.
// min_overlap <= 0 is tile-dependent in the reference (touching records count only when co-tiled) and is rejected.
#include <algorithm>
#include <condition_variable>
#include <cstdlib>
#include <map>
#include <memory>
#include <numeric>

#include "common.cuh"

namespace gtgpu {

namespace {

template <class T>
int32_t dev_alloc(gtgpu_igd* g, uint64_t count, T** out) {
    void* d = nullptr;
    size_t bytes = std::max<size_t>(count * sizeof(T), 16);
    cudaError_t e = cudaMalloc(&d, bytes);
    if (e != cudaSuccess) return fail(GTGPU_ERR_NOMEM, std::string("cudaMalloc(igd): ") + cudaGetErrorString(e));
    g->allocs.push_back(d);
    g->device_bytes += bytes;
    *out = (T*)d;
    return GTGPU_OK;
}

template <class T>
int32_t up(gtgpu_igd* g, const std::vector<T>& v, T** out) {
    GT_TRY(dev_alloc(g, v.size(), out));
    if (!v.empty()) GT_CUDA(cudaMemcpy(*out, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice));
    return GTGPU_OK;
}

// temporaries of a build: freed when the builder leaves
struct TempPool {
    std::vector<void*> ptrs;
    template <class T>
    int32_t get(uint64_t count, T** out) {
        void* d = nullptr;
        cudaError_t e = cudaMalloc(&d, std::max<size_t>(count * sizeof(T), 16));
        if (e != cudaSuccess) return fail(GTGPU_ERR_NOMEM, std::string("cudaMalloc(igd build): ") + cudaGetErrorString(e));
        ptrs.push_back(d);
        *out = (T*)d;
        return GTGPU_OK;
    }
    ~TempPool() {
        for (void* p : ptrs) cudaFree(p);
    }
};

int grid_for(const gtgpu_ctx* ctx, uint64_t n) {
    return (int)std::max<uint64_t>(1, std::min<uint64_t>((n + 255) / 256, (uint64_t)ctx->sm_count * 16));
}

}  // namespace

// ---- build kernels ---------------------------------------------------------------------------------------------------
// Sort key of an input record: its chromosome when Igd::add keeps it (igd.rs:109-116, 285-301: start < end as u32, then
// 0 <= start < end as i32), else n_chroms — dropped records sort behind every chromosome and are cut off.
__global__ void igd_chrom_keys_kernel(uint64_t n, uint32_t n_chroms, const uint32_t* __restrict__ chr, const uint32_t* __restrict__ start,
                                      const uint32_t* __restrict__ end, uint32_t* __restrict__ key) {
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        const uint32_t c = chr[i], s = start[i], e = end[i];
        const bool keep = c < n_chroms && s < e && (int32_t)s >= 0 && (int32_t)e >= 0;
        key[i] = keep ? c : n_chroms;
    }
}

// The .tsv statistics of every input file (Igd::from_named_region_sets, igd.rs:285-317): the region lines with start < end as
// u32 (dropped negative ones included) and the wrapping u64 sum of their widths (i32 end - i32 start, widened).  A file's records
// are contiguous, so a warp whose lanes share one file adds its sums once.
__global__ void igd_file_stats_kernel(uint64_t n, const uint32_t* __restrict__ start, const uint32_t* __restrict__ end,
                                      const uint32_t* __restrict__ file, unsigned long long* __restrict__ regions,
                                      unsigned long long* __restrict__ widths) {
    constexpr uint32_t FULL = 0xFFFFFFFFu;
    const uint32_t lane = threadIdx.x & 31;
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t base = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x - lane; base < n; base += stride) {
        const uint64_t i = base + lane;
        const bool ok = i < n;
        const uint32_t s = ok ? start[i] : 0, e = ok ? end[i] : 0, f = ok ? file[i] : 0;
        const bool region = ok && s < e;
        unsigned long long c = region, w = region ? (unsigned long long)(long long)(int32_t)(e - s) : 0ull;
        const uint32_t f0 = __shfl_sync(FULL, f, 0);  // lane 0 is always in range
        if (__all_sync(FULL, !ok || f == f0)) {
#pragma unroll
            for (int o = 16; o; o >>= 1) {
                c += __shfl_xor_sync(FULL, c, o);
                w += __shfl_xor_sync(FULL, w, o);
            }
            if (lane == 0 && c) {
                atomicAdd(regions + f0, c);
                atomicAdd(widths + f0, w);
            }
        } else if (region) {
            atomicAdd(regions + f, 1ull);
            atomicAdd(widths + f, w);
        }
    }
}

// first[c] = min over the kept records of chromosome c of their input index (file == nullptr) or their file.  chrkey is
// sorted, so a warp mostly holds one chromosome and reduces before its one atomic.
__global__ void igd_first_kept_kernel(uint64_t n, const uint32_t* __restrict__ chrkey, const uint32_t* __restrict__ perm,
                                      const uint32_t* __restrict__ file, uint32_t* __restrict__ first) {
    constexpr uint32_t FULL = 0xFFFFFFFFu;
    const uint32_t lane = threadIdx.x & 31;
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t base = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x - lane; base < n; base += stride) {
        const uint64_t k = base + lane;
        const bool ok = k < n;
        const uint32_t c = ok ? chrkey[k] : 0;
        uint32_t v = 0xFFFFFFFFu;
        if (ok) v = file ? file[perm[k]] : perm[k];
        const uint32_t c0 = __shfl_sync(FULL, c, 0);
        if (__all_sync(FULL, !ok || c == c0)) {
            v = __reduce_min_sync(FULL, v);
            if (lane == 0) atomicMin(first + c0, v);
        } else if (ok) {
            atomicMin(first + c, v);
        }
    }
}

// packed[k] = segment << 32 | value: the running maximum of the low word inside a segment is a plain 64-bit max-scan
__global__ void igd_pack_pmax_kernel(uint64_t n, const uint32_t* __restrict__ chrkey, const int32_t* __restrict__ end,
                                     unsigned long long* __restrict__ packed) {
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t k = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; k < n; k += stride)
        packed[k] = ((unsigned long long)chrkey[k] << 32) | (uint32_t)end[k];
}
__global__ void igd_low_words_kernel(uint64_t n, const unsigned long long* __restrict__ packed, int32_t* __restrict__ out) {
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t k = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; k < n; k += stride) out[k] = (int32_t)(uint32_t)packed[k];
}

// Records in (chromosome, file, pooled position) order: head[k] = 1 where a (chromosome, file) group starts
__global__ void igd_group_heads_kernel(uint64_t n, const uint32_t* __restrict__ order, const uint32_t* __restrict__ chrkey,
                                       const uint32_t* __restrict__ file, uint32_t* __restrict__ head) {
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t k = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; k < n; k += stride) {
        uint32_t h = 1;
        if (k) {
            const uint32_t a = order[k], b = order[k - 1];
            h = chrkey[a] != chrkey[b] || file[a] != file[b];
        }
        head[k] = h;
    }
}
// packed[k] = group number << 32 | (end + 1 when the record is at least m long, else 0)
__global__ void igd_pack_psame_kernel(uint64_t n, const uint32_t* __restrict__ order, const uint32_t* __restrict__ head,
                                      const uint32_t* __restrict__ groups_before, const int32_t* __restrict__ start,
                                      const int32_t* __restrict__ end, int32_t m, unsigned long long* __restrict__ packed) {
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t k = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; k < n; k += stride) {
        const uint32_t i = order[k];
        const int32_t s = start[i], e = end[i];
        const uint32_t v = (e - s >= m) ? (uint32_t)e + 1u : 0u;
        packed[k] = ((unsigned long long)(groups_before[k] + head[k]) << 32) | v;
    }
}
// psame of the k-th record of a group = the running maximum up to its predecessor in the group (-1: none)
__global__ void igd_scatter_psame_kernel(uint64_t n, const uint32_t* __restrict__ order, const uint32_t* __restrict__ head,
                                         const unsigned long long* __restrict__ running, int32_t* __restrict__ psame) {
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t k = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; k < n; k += stride)
        psame[order[k]] = head[k] ? -1 : (int32_t)(uint32_t)running[k - 1] - 1;
}

int32_t launch_fill_set_ids(gtgpu_ctx* ctx, uint64_t n_sets, const uint64_t* d_set_offsets, uint32_t* d_set_of);

namespace {

// psame[i] = max end over EARLIER records (pooled order) of the same file on the same chromosome with end - start >= m;
// -1 when there is none.  Pooled positions are regrouped by (chromosome, file) with two stable radix passes, the running
// maximum inside a group is one max-scan, and the result goes back to the pooled positions.
int32_t device_psame(gtgpu_igd* g, int32_t m, int32_t* d_psame) {
    gtgpu_ctx* ctx = g->ctx;
    const uint64_t n = g->n_records;
    if (n == 0) return GTGPU_OK;
    cudaStream_t st = ctx->stream;
    TempPool tp;
    uint32_t *d_chrkey, *d_head, *d_before;
    uint64_t* d_off64;
    unsigned long long* d_packed;
    char* d_scan_tmp;
    GT_TRY(tp.get(n, &d_chrkey));
    GT_TRY(tp.get(n, &d_head));
    GT_TRY(tp.get(n, &d_before));
    GT_TRY(tp.get(g->n_chroms + 1, &d_off64));
    GT_TRY(tp.get(n, &d_packed));
    GT_TRY(tp.get(exclusive_scan_temp_bytes(n, 8), &d_scan_tmp));
    std::vector<uint64_t> off64(g->h_off.begin(), g->h_off.end());
    GT_CUDA(cudaMemcpyAsync(d_off64, off64.data(), off64.size() * 8, cudaMemcpyHostToDevice, st));
    GT_CUDA(cudaStreamSynchronize(st));
    GT_TRY(launch_fill_set_ids(ctx, g->n_chroms, d_off64, d_chrkey));
    PermSorter by_group;
    GT_TRY(by_group.init(ctx, n));
    GT_TRY(by_group.pass(g->d_file, bits_for_value(g->n_files ? g->n_files - 1 : 0)));
    GT_TRY(by_group.pass(d_chrkey, bits_for_value(g->n_chroms)));
    const int grid = grid_for(ctx, n);
    igd_group_heads_kernel<<<grid, 256, 0, st>>>(n, by_group.perm, d_chrkey, g->d_file, d_head);
    GT_TRY(exclusive_scan<uint32_t>(ctx, d_head, d_before, n, d_scan_tmp));
    igd_pack_psame_kernel<<<grid, 256, 0, st>>>(n, by_group.perm, d_head, d_before, g->d_start, g->d_end, m, d_packed);
    GT_TRY(inclusive_max_scan_u64(ctx, d_packed, d_packed, n, d_scan_tmp));
    igd_scatter_psame_kernel<<<grid, 256, 0, st>>>(n, by_group.perm, d_head, d_packed, d_psame);
    ctx->launches += 3;
    GT_CUDA(cudaGetLastError());
    GT_CUDA(cudaStreamSynchronize(st));
    return GTGPU_OK;
}

}  // namespace

// Warp-cooperative lower bound (first index whose value is >= key) inside [lo, hi): 32 probes per step instead of one.
// A bisection costs log2(range) DEPENDENT loads, and with one query per warp that chain — two searches of five to eight
// round trips each — was most of a query's time: nothing in the memory system was more than 60 % busy (ncu, C4).
__device__ __forceinline__ uint32_t lb_warp(const int32_t* __restrict__ arr, uint32_t lo, uint32_t hi, int32_t key, uint32_t lane) {
    constexpr uint32_t FULL = 0xFFFFFFFFu;
    while (hi - lo > 32u) {  // 32 evenly spaced samples: the answer lies between two neighbours
        const uint32_t step = (hi - lo + 31u) / 32u, idx = lo + lane * step;
        const bool below = idx < hi && __ldg(arr + idx) < key;
        const uint32_t k = __popc(__ballot_sync(FULL, below));  // the samples are sorted: the first k are below the key
        if (k == 0) return lo;
        const uint32_t first = lo + (k - 1) * step + 1;
        hi = min(lo + k * step, hi);
        lo = first;
    }
    const bool below = lo + lane < hi && __ldg(arr + lo + lane) < key;
    return lo + __popc(__ballot_sync(FULL, below));
}

struct IgdView {
    const uint32_t *off, *lut_s_off, *nb_s, *lut_p_off, *nb_p, *file, *lut;
    const int32_t *start, *end, *pmax, *psame;
    uint32_t n_chroms, shift;
    uint64_t n_files;
};

// One warp per query.  BINARY selects count_region_hits semantics.
#ifndef GT_IGD_MINBLOCKS
#define GT_IGD_MINBLOCKS 5
#endif
#ifndef GT_IGD_MINBLOCKS_M1
#define GT_IGD_MINBLOCKS_M1 6
#endif
// M1: min_overlap == 1 (LOLA's and every reference caller's setting).  Every candidate already starts before the query's end,
// and a stored record has start < end, so it overlaps by at least one base iff it ends after the query's start: the start
// array is not read at all — 12 instead of 16 bytes per candidate of a kernel that pulls 72 GB of records from DRAM on C4.
template <bool BINARY, bool M1>
__global__ void __launch_bounds__(256, M1 ? GT_IGD_MINBLOCKS_M1 : GT_IGD_MINBLOCKS) igd_count_kernel(IgdView v, uint64_t n, const uint32_t* __restrict__ set_of,
                                                         const uint32_t* __restrict__ chr, const uint32_t* __restrict__ qstart,
                                                         const uint32_t* __restrict__ qend, int32_t m,
                                                         unsigned long long* __restrict__ out) {
    const uint32_t lane = threadIdx.x & 31;
    const uint64_t warps = ((uint64_t)gridDim.x * blockDim.x) >> 5;
    uint64_t q = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    // the next query (and its set) is requested while this one is resolved
    uint32_t nc = 0, nset = 0;
    int32_t ns = 0, ne = 0;
    if (q < n) {
        nc = __ldg(chr + q);
        ns = (int32_t)__ldg(qstart + q);
        ne = (int32_t)__ldg(qend + q);
        nset = __ldg(set_of + q);
    }
    for (; q < n; q += warps) {
        const uint32_t c = nc, set = nset;
        int32_t s = ns, e = ne;
        if (q + warps < n) {
            nc = __ldg(chr + q + warps);
            ns = (int32_t)__ldg(qstart + q + warps);
            ne = (int32_t)__ldg(qend + q + warps);
            nset = __ldg(set_of + q + warps);
        }
        if (c >= v.n_chroms || s >= e || e <= 0) continue;  // igd.rs:514-522
        s = max(s, 0);
        const uint32_t o = __ldg(v.off + c), len = __ldg(v.off + c + 1) - o;
        if (len == 0) continue;
        // records that can reach the query: start < e, and some record at or before them ends after s.  Both searches start
        // from their LUT bins (four independent loads), then narrow 32 probes at a time.
        const uint32_t* lut_s = v.lut + __ldg(v.lut_s_off + c);
        const uint32_t* lut_p = v.lut + __ldg(v.lut_p_off + c);
        const uint32_t nb_s = __ldg(v.nb_s + c), nb_p = __ldg(v.nb_p + c);
        const uint32_t bs = (uint32_t)e >> v.shift, bp = (uint32_t)(s + 1) >> v.shift;  // e >= 1, s + 1 >= 1
        uint32_t s_lo = len, s_hi = len, p_lo = len, p_hi = len;
        if (bs < nb_s) {
            s_lo = __ldg(lut_s + bs);
            s_hi = __ldg(lut_s + bs + 1);
        }
        if (bp < nb_p) {
            p_lo = __ldg(lut_p + bp);
            p_hi = __ldg(lut_p + bp + 1);
        }
        const uint32_t ub = lb_warp(v.start + o, s_lo, s_hi, e, lane);
        const uint32_t lo = lb_warp(v.pmax + o, p_lo, p_hi, s + 1, lane);
        unsigned long long* row = out + (uint64_t)set * v.n_files;
        // 128 candidates per round: every lane requests its four records (start, end, file, psame — sixteen independent loads)
        // before it tests any of them: 24.7 -> 18.9 ms on the LOLA configuration (1 k x 10 k sets).  ncu (profiles/r02/
        // c4_igd_count_ncu_full.txt): the reductions run at a quarter of the L2's rate; the kernel waits on its own chain of
        // loads per query with the memory system at half load (72 GB of record reads from DRAM).  Walking the queries in
        // genome order (radix-sorted) did not change the kernel time (18.4 ms), and a variant that kept the current set's
        // matrix row in shared memory (32-bit shared atomics, one flush per 4 096 queries) was slower (41 ms) — both measured
        // in round 2 and dropped.
        for (uint32_t base = o + lo; base < o + ub; base += 128) {
            int32_t rs[4], re[4], ps[4];
            uint32_t fl[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const uint32_t i = base + 32 * k + lane;
                const bool ok = i < o + ub;
                rs[k] = (!M1 && ok) ? __ldg(v.start + i) : 0;
                re[k] = ok ? __ldg(v.end + i) : 0;  // an absent record [0, 0) never reaches m >= 1 bp of overlap (s >= 0)
                fl[k] = ok ? __ldg(v.file + i) : 0;
                ps[k] = (BINARY && ok) ? __ldg(v.psame + i) : 0;
            }
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                if (M1 ? re[k] <= s : min(re[k], e) - max(rs[k], s) < m) continue;
                if (BINARY && (int64_t)ps[k] - s >= m) continue;  // an earlier record of this file already hit
                atomicAdd(row + fl[k], 1ull);
            }
        }
    }
}

// set index of every query from the set offsets (one thread per set writes its range)
__global__ void fill_set_ids_kernel(uint64_t n_sets, const uint64_t* __restrict__ set_offsets, uint32_t* __restrict__ set_of) {
    for (uint64_t s = blockIdx.x; s < n_sets; s += gridDim.x)
        for (uint64_t i = set_offsets[s] + threadIdx.x; i < set_offsets[s + 1]; i += blockDim.x) set_of[i] = (uint32_t)s;
}

int32_t launch_fill_set_ids(gtgpu_ctx* ctx, uint64_t n_sets, const uint64_t* d_set_offsets, uint32_t* d_set_of) {
    if (!n_sets) return GTGPU_OK;
    fill_set_ids_kernel<<<(unsigned)std::min<uint64_t>(n_sets, 4096), 256, 0, ctx->stream>>>(n_sets, d_set_offsets, d_set_of);
    ctx->launches++;
    GT_CUDA(cudaGetLastError());
    return GTGPU_OK;
}

}  // namespace gtgpu

using namespace gtgpu;

// Multi-device group: the database is sharded by region set (run_lola's database axis, enrichment.rs:198-211): device r
// builds its own record pool over sets [r * C, min((r + 1) * C, n_files)), C = ceil(n_files / devices), all in parallel.
// contig_by_file: the records come from BED files, whose RegionSets the reference sorts by (name, start) before Igd::add sees them
// (gtgpu_igd_serialize's contig order).
static int32_t igd_build_one(gtgpu_ctx* ctx, uint64_t n_files, const uint64_t* file_offsets, uint32_t n_chroms, const uint32_t* chr,
                             const uint32_t* start, const uint32_t* end, bool contig_by_file, gtgpu_igd** out_igd);
static int32_t igd_build_dev(gtgpu_ctx* ctx, uint64_t n_files, uint32_t n_chroms, uint64_t total, const uint32_t* t_chr,
                             const uint32_t* t_start, const uint32_t* t_end, const uint32_t* t_file, bool contig_by_file,
                             gtgpu_igd** out_igd);

static int32_t igd_build_group(gtgpu_ctx* ctx, uint64_t n_files, const uint64_t* file_offsets, uint32_t n_chroms, const uint32_t* chr,
                               const uint32_t* start, const uint32_t* end, bool contig_by_file, gtgpu_igd** out_igd) {
    std::lock_guard<std::mutex> glk(ctx->group_mu);
    const size_t D = ctx->peers.size();
    const uint64_t cols = (n_files + D - 1) / D;
    std::unique_ptr<gtgpu_igd> g(new gtgpu_igd());
    g->ctx = ctx;
    g->n_files = n_files;
    g->n_chroms = n_chroms;
    g->shards.assign(D, nullptr);
    const int32_t s = for_each_device(D, [&](size_t r) -> int32_t {
        const uint64_t lo = std::min<uint64_t>(r * cols, n_files), hi = std::min<uint64_t>(lo + cols, n_files);
        std::vector<uint64_t> fo(hi - lo + 1);
        for (uint64_t f = lo; f <= hi; ++f) fo[f - lo] = file_offsets[f] - file_offsets[lo];
        const uint64_t r0 = file_offsets[lo];
        // (peers[0] is the group context itself: the single-device builder is called directly, not through the entry point)
        const int32_t st = igd_build_one(ctx->peers[r], hi - lo, fo.data(), n_chroms, chr ? chr + r0 : nullptr,
                                         start ? start + r0 : nullptr, end ? end + r0 : nullptr, contig_by_file, &g->shards[r]);
        if (st == GTGPU_OK) {
            g->shards[r]->file0 = lo;
            g->shards[r]->rec0 = r0;
        }
        return st;
    });
    if (s != GTGPU_OK) {
        const std::string msg = gtgpu_last_error();
        for (auto* sh : g->shards) gtgpu_igd_free(sh);
        return fail(s, msg);
    }
    for (auto* sh : g->shards) {
        g->n_records += sh->n_records;
        g->device_bytes += sh->device_bytes;
    }
    g->shift = g->shards[0]->shift;
    g->contig_by_file = contig_by_file;
    *out_igd = g.release();
    return GTGPU_OK;
}

extern "C" int32_t gtgpu_igd_build(gtgpu_ctx* ctx, uint64_t n_files, const uint64_t* file_offsets, uint32_t n_chroms,
                                   const uint32_t* chr, const uint32_t* start, const uint32_t* end, gtgpu_igd** out_igd) try {
    if (!ctx || !out_igd || !file_offsets) return fail(GTGPU_ERR_INVALID, "igd_build: null argument");
    for (uint64_t f = 0; f < n_files; ++f)
        if (file_offsets[f] > file_offsets[f + 1]) return fail(GTGPU_ERR_INVALID, "igd_build: file_offsets not monotone");
    if (file_offsets[0] != 0) return fail(GTGPU_ERR_INVALID, "igd_build: file_offsets[0] must be 0");
    const uint64_t total = file_offsets[n_files];
    if (total && (!chr || !start || !end)) return fail(GTGPU_ERR_INVALID, "igd_build: null record arrays");
    if (total >= 0xFFFFFFFFull || n_files >= 0xFFFFFFFFull || n_chroms >= 0x7FFFFFFFu)
        return fail(GTGPU_ERR_UNSUPPORTED, "igd_build: too many records");
    if (ctx->peers.size() > 1) return igd_build_group(ctx, n_files, file_offsets, n_chroms, chr, start, end, false, out_igd);
    return igd_build_one(ctx, n_files, file_offsets, n_chroms, chr, start, end, false, out_igd);
} GT_CATCH

// ---- a database from its BED files' text, parsed on the device --------------------------------------------------------------
// The records and the chromosome names come from parse_bed_files_locked on ctx (the first device of a group).  One device: the
// build reads the parsed records where they are.  A group: shard r's files are a contiguous record range, copied to its
// device with cudaMemcpyAsync by the builder of gtgpu_igd_build (igd_records_to_device).
static int32_t igd_build_parsed(gtgpu_ctx* ctx, uint64_t n_files, BedFilesRecords& r, uint32_t* out_n_chroms, gtgpu_buf** out_names,
                                gtgpu_buf** out_name_offsets, gtgpu_igd** out_igd) {
    const uint32_t n_chroms = r.n_names;
    gtgpu_igd* g = nullptr;
    if (ctx->peers.size() > 1) {
        GT_TRY(igd_build_group(ctx, n_files, r.file_offsets.data(), n_chroms, r.chr.u32(), r.start.u32(), r.end.u32(), true, &g));
        GT_CUDA(cudaSetDevice(ctx->device));  // the parsed records are freed on their device
    } else {
        std::lock_guard<std::mutex> lk(ctx->mu);
        GT_CUDA(cudaSetDevice(ctx->device));
        GT_TRY(igd_build_dev(ctx, n_files, n_chroms, r.n, r.chr.u32(), r.start.u32(), r.end.u32(), r.file.u32(), true, &g));
    }
    *out_n_chroms = n_chroms;
    *out_names = r.names.release();
    *out_name_offsets = r.name_offsets.release();
    *out_igd = g;
    return GTGPU_OK;
}

extern "C" int32_t gtgpu_igd_build_bed(gtgpu_ctx* ctx, uint64_t n_files, const char* text, const uint64_t* file_offsets,
                                       uint32_t* out_n_chroms, gtgpu_buf** out_chrom_names, gtgpu_buf** out_chrom_name_offsets,
                                       gtgpu_igd** out_igd) try {
    if (!ctx || !file_offsets || !out_n_chroms || !out_chrom_names || !out_chrom_name_offsets || !out_igd)
        return fail(GTGPU_ERR_INVALID, "igd_build_bed: null argument");
    if (file_offsets[0] != 0) return fail(GTGPU_ERR_INVALID, "igd_build_bed: file_offsets[0] must be 0");
    for (uint64_t f = 0; f < n_files; ++f)
        if (file_offsets[f] > file_offsets[f + 1]) return fail(GTGPU_ERR_INVALID, "igd_build_bed: file_offsets not monotone");
    if (file_offsets[n_files] && !text) return fail(GTGPU_ERR_INVALID, "igd_build_bed: null text");
    if (n_files >= 0xFFFFFFFFull) return fail(GTGPU_ERR_UNSUPPORTED, "igd_build_bed: too many files");
    BedFilesRecords r;
    {
        std::lock_guard<std::mutex> lk(ctx->mu);
        GT_CUDA(cudaSetDevice(ctx->device));
        GT_TRY(parse_bed_files_locked(ctx, text, nullptr, n_files, file_offsets, "igd_build_bed", &r));
    }
    return igd_build_parsed(ctx, n_files, r, out_n_chroms, out_chrom_names, out_chrom_name_offsets, out_igd);
} GT_CATCH

extern "C" int32_t gtgpu_igd_build_bed_gz(gtgpu_ctx* ctx, uint64_t n_files, const uint64_t* file_members, uint64_t n_members,
                                          const uint8_t* gz, const uint64_t* member_offsets, uint32_t* out_n_chroms,
                                          gtgpu_buf** out_chrom_names, gtgpu_buf** out_chrom_name_offsets, gtgpu_igd** out_igd) try {
    if (!ctx || !file_members || !out_n_chroms || !out_chrom_names || !out_chrom_name_offsets || !out_igd)
        return fail(GTGPU_ERR_INVALID, "igd_build_bed_gz: null argument");
    GT_TRY(check_members(n_members, gz, member_offsets, "igd_build_bed_gz"));
    if (file_members[0] != 0 || file_members[n_files] != n_members)
        return fail(GTGPU_ERR_INVALID, "igd_build_bed_gz: file_members must run from 0 to n_members");
    for (uint64_t f = 0; f < n_files; ++f)
        if (file_members[f] > file_members[f + 1]) return fail(GTGPU_ERR_INVALID, "igd_build_bed_gz: file_members not monotone");
    if (n_files >= 0xFFFFFFFFull) return fail(GTGPU_ERR_UNSUPPORTED, "igd_build_bed_gz: too many files");
    BedFilesRecords r;
    {
        std::lock_guard<std::mutex> lk(ctx->mu);
        GT_CUDA(cudaSetDevice(ctx->device));
        uint8_t* d_text = nullptr;
        uint64_t n_text = 0;
        std::vector<uint64_t> text_offsets(n_members + 1), fo(n_files + 1);
        GT_TRY(inflate_whole_locked(ctx, n_members, gz, member_offsets, "igd_build_bed_gz", &d_text, &n_text, text_offsets.data()));
        for (uint64_t f = 0; f <= n_files; ++f) fo[f] = text_offsets[file_members[f]];
        GT_TRY(parse_bed_files_locked(ctx, nullptr, (const char*)d_text, n_files, fo.data(), "igd_build_bed_gz", &r));
    }
    return igd_build_parsed(ctx, n_files, r, out_n_chroms, out_chrom_names, out_chrom_name_offsets, out_igd);
} GT_CATCH

// Records to the device: chr / start / end (host or device memory, any device: cudaMemcpyDefault) into temporaries of tp, and
// every record's file index from file_offsets.
static int32_t igd_records_to_device(gtgpu_ctx* ctx, TempPool& tp, uint64_t n_files, const uint64_t* file_offsets, const uint32_t* chr,
                                     const uint32_t* start, const uint32_t* end, uint32_t** t_chr, uint32_t** t_start, uint32_t** t_end,
                                     uint32_t** t_file) {
    const uint64_t total = file_offsets[n_files];
    cudaStream_t st = ctx->stream;
    uint64_t* t_fo;
    GT_TRY(tp.get(total, t_chr));
    GT_TRY(tp.get(total, t_start));
    GT_TRY(tp.get(total, t_end));
    GT_TRY(tp.get(total, t_file));
    GT_TRY(tp.get(n_files + 1, &t_fo));
    if (total) {
        GT_CUDA(cudaMemcpyAsync(*t_chr, chr, total * 4, cudaMemcpyDefault, st));
        GT_CUDA(cudaMemcpyAsync(*t_start, start, total * 4, cudaMemcpyDefault, st));
        GT_CUDA(cudaMemcpyAsync(*t_end, end, total * 4, cudaMemcpyDefault, st));
    }
    GT_CUDA(cudaMemcpyAsync(t_fo, file_offsets, (n_files + 1) * 8, cudaMemcpyHostToDevice, st));
    GT_CUDA(cudaStreamSynchronize(st));  // the caller's arrays may be pageable
    if (total) GT_TRY(launch_fill_set_ids(ctx, n_files, t_fo, *t_file));
    return GTGPU_OK;
}

static int32_t igd_build_one(gtgpu_ctx* ctx, uint64_t n_files, const uint64_t* file_offsets, uint32_t n_chroms, const uint32_t* chr,
                             const uint32_t* start, const uint32_t* end, bool contig_by_file, gtgpu_igd** out_igd) {
    std::lock_guard<std::mutex> lk(ctx->mu);
    GT_CUDA(cudaSetDevice(ctx->device));
    TempPool tp;
    uint32_t *t_chr, *t_start, *t_end, *t_file;
    GT_TRY(igd_records_to_device(ctx, tp, n_files, file_offsets, chr, start, end, &t_chr, &t_start, &t_end, &t_file));
    return igd_build_dev(ctx, n_files, n_chroms, file_offsets[n_files], t_chr, t_start, t_end, t_file, contig_by_file, out_igd);
}

// The build from device-resident records of this ctx's device (record i belongs to file t_file[i]).  The caller holds ctx->mu.
static int32_t igd_build_dev(gtgpu_ctx* ctx, uint64_t n_files, uint32_t n_chroms, uint64_t total, const uint32_t* t_chr,
                             const uint32_t* t_start, const uint32_t* t_end, const uint32_t* t_file, bool contig_by_file,
                             gtgpu_igd** out_igd) {
    cudaStream_t st = ctx->stream;
    gtgpu_igd* g = new gtgpu_igd();
    g->ctx = ctx;
    g->n_files = n_files;
    g->n_chroms = n_chroms;
    g->contig_by_file = contig_by_file;
    struct Guard {  // a failed build frees what it allocated
        gtgpu_igd* g;
        ~Guard() { if (g) gtgpu_igd_free(g); }
    } guard{g};

    // ---- 1. pooled order = stable sort by (chromosome, start) -------------------------------------------------------
    // ties keep (file, insertion) order = the order Igd::add saw them (igd.rs:285-301); records Igd::add drops get the
    // key n_chroms, land behind the last chromosome and are cut off
    TempPool tp;
    uint32_t *t_key, *t_off;
    GT_TRY(tp.get(total, &t_key));
    GT_TRY(tp.get(n_chroms + 2, &t_off));
    PermSorter pooled;
    GT_TRY(pooled.init(ctx, total));
    if (total) {
        igd_chrom_keys_kernel<<<grid_for(ctx, total), 256, 0, st>>>(total, n_chroms, t_chr, t_start, t_end, t_key);
        ctx->launches++;
        GT_TRY(pooled.pass(t_start, 0));
        GT_TRY(pooled.pass(t_key, bits_for_value(n_chroms)));
    }
    g->h_off.assign(n_chroms + 1, 0);
    if (total) {
        GT_TRY(launch_key_offsets(ctx, total, pooled.key, n_chroms, t_off));
        GT_CUDA(cudaMemcpyAsync(g->h_off.data(), t_off, (n_chroms + 1) * 4, cudaMemcpyDeviceToHost, st));
        GT_CUDA(cudaStreamSynchronize(st));
    }
    const uint64_t n_rec = g->h_off[n_chroms];
    g->n_records = n_rec;

    // ---- what a save needs besides the records: the .tsv statistics of every file, the first kept record of every chromosome
    {
        unsigned long long* d_stats;
        uint32_t* d_first;
        GT_TRY(tp.get(2 * n_files, &d_stats));
        GT_TRY(tp.get(n_chroms, &d_first));
        if (n_files) GT_CUDA(cudaMemsetAsync(d_stats, 0, 2 * n_files * 8, st));
        if (n_chroms) GT_CUDA(cudaMemsetAsync(d_first, 0xFF, (uint64_t)n_chroms * 4, st));
        if (total) {
            igd_file_stats_kernel<<<grid_for(ctx, total), 256, 0, st>>>(total, t_start, t_end, t_file, d_stats, d_stats + n_files);
            ctx->launches++;
        }
        if (n_rec) {
            igd_first_kept_kernel<<<grid_for(ctx, n_rec), 256, 0, st>>>(n_rec, pooled.key, pooled.perm, contig_by_file ? t_file : nullptr,
                                                                        d_first);
            ctx->launches++;
        }
        GT_CUDA(cudaGetLastError());
        g->h_file_regions.assign(n_files, 0);
        g->h_file_widths.assign(n_files, 0);
        g->h_first.assign(n_chroms, 0xFFFFFFFFu);
        if (n_files) {
            GT_CUDA(cudaMemcpyAsync(g->h_file_regions.data(), d_stats, n_files * 8, cudaMemcpyDeviceToHost, st));
            GT_CUDA(cudaMemcpyAsync(g->h_file_widths.data(), d_stats + n_files, n_files * 8, cudaMemcpyDeviceToHost, st));
        }
        if (n_chroms) GT_CUDA(cudaMemcpyAsync(g->h_first.data(), d_first, (uint64_t)n_chroms * 4, cudaMemcpyDeviceToHost, st));
        GT_CUDA(cudaStreamSynchronize(st));
    }

    // ---- 2. the kept records in pooled order, running max of ends per chromosome ------------------------------------
    GT_TRY(dev_alloc(g, n_rec, &g->d_start));
    GT_TRY(dev_alloc(g, n_rec, &g->d_end));
    GT_TRY(dev_alloc(g, n_rec, &g->d_file));
    GT_TRY(dev_alloc(g, n_rec, &g->d_pmax));
    GT_TRY(dev_alloc(g, n_rec, &g->d_psame1));
    std::vector<uint32_t> last_start(n_chroms, 0), last_pmax(n_chroms, 0);
    if (n_rec) {
        GT_TRY(launch_gather_u32(ctx, n_rec, t_start, pooled.perm, (uint32_t*)g->d_start));
        GT_TRY(launch_gather_u32(ctx, n_rec, t_end, pooled.perm, (uint32_t*)g->d_end));
        GT_TRY(launch_gather_u32(ctx, n_rec, t_file, pooled.perm, g->d_file));
        unsigned long long* d_packed;
        char* d_scan_tmp;
        GT_TRY(tp.get(n_rec, &d_packed));
        GT_TRY(tp.get(exclusive_scan_temp_bytes(n_rec, 8), &d_scan_tmp));
        igd_pack_pmax_kernel<<<grid_for(ctx, n_rec), 256, 0, st>>>(n_rec, pooled.key, g->d_end, d_packed);
        GT_TRY(inclusive_max_scan_u64(ctx, d_packed, d_packed, n_rec, d_scan_tmp));
        igd_low_words_kernel<<<grid_for(ctx, n_rec), 256, 0, st>>>(n_rec, d_packed, g->d_pmax);
        ctx->launches += 2;
        GT_CUDA(cudaGetLastError());
        // the last start / running max of every chromosome size the LUTs
        for (uint32_t c = 0; c < n_chroms; ++c) {
            if (g->h_off[c + 1] == g->h_off[c]) continue;
            GT_CUDA(cudaMemcpyAsync(&last_start[c], g->d_start + g->h_off[c + 1] - 1, 4, cudaMemcpyDeviceToHost, st));
            GT_CUDA(cudaMemcpyAsync(&last_pmax[c], g->d_pmax + g->h_off[c + 1] - 1, 4, cudaMemcpyDeviceToHost, st));
        }
        GT_CUDA(cudaStreamSynchronize(st));
    }
    g->h_max_end = last_pmax;

    // ---- 3. bin LUTs over starts and running maxima: at most ~8 M bins per family --------------------------------------
    uint32_t shift = 0;
    auto bins = [&](uint32_t sh) {
        uint64_t t = 0;
        for (uint32_t c = 0; c < n_chroms; ++c)
            if (g->h_off[c + 1] > g->h_off[c]) t += (last_pmax[c] >> sh) + 2;
        return t;
    };
    const uint64_t budget = std::min<uint64_t>(std::max<uint64_t>(n_rec, 4096), 8ull << 20);
    while (shift < 31 && bins(shift) > budget) ++shift;
    g->shift = shift;
    std::vector<uint32_t> lso(n_chroms), nbs(n_chroms), lpo(n_chroms), nbp(n_chroms);
    std::vector<LutDesc> desc_s(n_chroms), desc_p(n_chroms);
    std::vector<uint64_t> pre_s(n_chroms + 1, 0), pre_p(n_chroms + 1, 0);
    uint64_t lut_len = 0;
    for (uint32_t c = 0; c < n_chroms; ++c) {
        const uint32_t o = g->h_off[c], len = g->h_off[c + 1] - o;
        nbs[c] = len ? (last_start[c] >> shift) + 1 : 0;
        nbp[c] = len ? (last_pmax[c] >> shift) + 1 : 0;
        lso[c] = (uint32_t)lut_len;
        lut_len += (uint64_t)nbs[c] + 1;
        lpo[c] = (uint32_t)lut_len;
        lut_len += (uint64_t)nbp[c] + 1;
        desc_s[c] = LutDesc{o, len, lso[c], nbs[c]};
        desc_p[c] = LutDesc{o, len, lpo[c], nbp[c]};
        pre_s[c + 1] = pre_s[c] + nbs[c] + 1;
        pre_p[c + 1] = pre_p[c] + nbp[c] + 1;
    }
    if (lut_len >= 0xFFFFFFFFull) return fail(GTGPU_ERR_UNSUPPORTED, "igd_build: LUT too large");
    GT_TRY(dev_alloc(g, lut_len, &g->d_lut));
    if (n_chroms) {
        LutDesc *d_desc_s, *d_desc_p;
        uint64_t *d_pre_s, *d_pre_p;
        GT_TRY(tp.get(n_chroms, &d_desc_s));
        GT_TRY(tp.get(n_chroms, &d_desc_p));
        GT_TRY(tp.get(n_chroms + 1, &d_pre_s));
        GT_TRY(tp.get(n_chroms + 1, &d_pre_p));
        GT_CUDA(cudaMemcpyAsync(d_desc_s, desc_s.data(), n_chroms * sizeof(LutDesc), cudaMemcpyHostToDevice, st));
        GT_CUDA(cudaMemcpyAsync(d_desc_p, desc_p.data(), n_chroms * sizeof(LutDesc), cudaMemcpyHostToDevice, st));
        GT_CUDA(cudaMemcpyAsync(d_pre_s, pre_s.data(), (n_chroms + 1) * 8, cudaMemcpyHostToDevice, st));
        GT_CUDA(cudaMemcpyAsync(d_pre_p, pre_p.data(), (n_chroms + 1) * 8, cudaMemcpyHostToDevice, st));
        GT_TRY(launch_build_luts(ctx, n_chroms, d_desc_s, d_pre_s, pre_s[n_chroms], (const uint32_t*)g->d_start, shift, g->d_lut));
        GT_TRY(launch_build_luts(ctx, n_chroms, d_desc_p, d_pre_p, pre_p[n_chroms], (const uint32_t*)g->d_pmax, shift, g->d_lut));
        GT_CUDA(cudaStreamSynchronize(st));  // the descriptor vectors are pageable
    }
    GT_TRY(device_psame(g, 1, g->d_psame1));
    GT_TRY(up(g, g->h_off, &g->d_off));
    GT_TRY(up(g, lso, &g->d_lut_s_off));
    GT_TRY(up(g, nbs, &g->d_nb_s));
    GT_TRY(up(g, lpo, &g->d_lut_p_off));
    GT_TRY(up(g, nbp, &g->d_nb_p));
    GT_CUDA(cudaStreamSynchronize(st));
    g->psame_by_m[1] = g->d_psame1;
    guard.g = nullptr;
    *out_igd = g;
    return GTGPU_OK;
}

extern "C" int32_t gtgpu_igd_free(gtgpu_igd* g) try {
    if (!g) return GTGPU_OK;
    for (gtgpu_igd* sh : g->shards) gtgpu_igd_free(sh);
    cudaSetDevice(g->ctx->device);
    for (void* p : g->allocs) cudaFree(p);
    delete g;
    return GTGPU_OK;
} GT_CATCH

extern "C" int32_t gtgpu_igd_info(const gtgpu_igd* g, uint64_t info[4]) try {
    if (!g || !info) return fail(GTGPU_ERR_INVALID, "igd_info: null argument");
    info[0] = g->n_files;
    info[1] = g->n_records;
    info[2] = g->device_bytes;
    info[3] = g->shift;
    return GTGPU_OK;
} GT_CATCH

namespace {

}  // namespace

namespace gtgpu {
int32_t igd_count_dev_locked(gtgpu_igd* g, bool binary, uint64_t n, const uint32_t* d_set_of, const uint32_t* d_chr,
                           const uint32_t* d_start, const uint32_t* d_end, int32_t m, uint64_t* d_out) {
    gtgpu_ctx* ctx = g->ctx;
    if (m < 1)
        return fail(GTGPU_ERR_UNSUPPORTED,
                    "igd count: min_overlap < 1 depends on the reference's tile layout (igd.rs:786-795) and is not supported");
    const int32_t* d_psame = nullptr;
    if (binary) {
        auto it = g->psame_by_m.find(m);
        if (it == g->psame_by_m.end()) {
            int32_t* d = nullptr;
            GT_TRY(dev_alloc(g, g->n_records, &d));
            GT_TRY(device_psame(g, m, d));
            it = g->psame_by_m.emplace(m, d).first;
        }
        d_psame = it->second;
    }
    if (n == 0) return GTGPU_OK;
    IgdView v{g->d_off, g->d_lut_s_off, g->d_nb_s, g->d_lut_p_off, g->d_nb_p, g->d_file, g->d_lut,
              g->d_start, g->d_end, g->d_pmax, d_psame, g->n_chroms, g->shift, g->n_files};
    // exactly the blocks that are resident at once (the queries are strided over the warps): a grid of 8 blocks per SM
    // ran a second, partial wave (17.3 vs 16.6 ms on C4); fewer resident warps are slower (4 per SM 17.8, 3: 21.3, 2: 28.9 ms),
    // and a sixth block per SM only fits with spills (21.9 ms)
    int ctas_per_sm = 0;
    const bool m1 = m == 1 && !(getenv("GTGPU_IGD_NO_M1") && *getenv("GTGPU_IGD_NO_M1") == '1');
    auto kern = binary ? (m1 ? igd_count_kernel<true, true> : igd_count_kernel<true, false>)
                       : (m1 ? igd_count_kernel<false, true> : igd_count_kernel<false, false>);
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ctas_per_sm, kern, 256, 0);
    if (ctas_per_sm < 1) ctas_per_sm = 4;
    if (const char* env = getenv("GTGPU_IGD_CTAS")) ctas_per_sm = std::max(1, atoi(env));  // tuning knob: blocks per SM of the grid
    const int grid = (int)std::min<uint64_t>((n + 7) / 8, (uint64_t)ctx->sm_count * ctas_per_sm);
    ctx->time_begin();
    kern<<<grid, 256, 0, ctx->stream>>>(v, n, d_set_of, d_chr, d_start, d_end, m, (unsigned long long*)d_out);
    ctx->time_end();
    ctx->launches++;
    GT_CUDA(cudaGetLastError());
    return GTGPU_OK;
}

// Group igd: every device counts the (replicated) query sets against its shard of the database, the column blocks are
// combined with ONE ncclAllGather between the devices (in-process communicators, NVLink), and the first device returns
// the [n_sets x n_files] matrix.  A barrier in front of the collective keeps device-memory allocation (implicitly
// synchronising) out of the window in which another device's collective kernel already waits for its peers.
int32_t igd_count_group(gtgpu_igd* g, bool binary, uint64_t n_sets, const uint64_t* set_offsets, const uint32_t* chr,
                        const uint32_t* start, const uint32_t* end, int32_t m, uint64_t* out) {
    gtgpu_ctx* ctx = g->ctx;
    std::lock_guard<std::mutex> glk(ctx->group_mu);
    GT_TRY(group_comm_ensure(ctx));
    const size_t D = g->shards.size();
    std::mutex bm;
    std::condition_variable bcv;
    size_t arrived = 0;
    bool all_ok = true;
    const std::function<bool(bool)> barrier = [&](bool ok) {
        std::unique_lock<std::mutex> l(bm);
        all_ok = all_ok && ok;
        if (++arrived == D) bcv.notify_all();
        else bcv.wait(l, [&] { return arrived == D; });
        return all_ok;
    };
    return for_each_device(D, [&](size_t r) -> int32_t {
        return igd_count_sharded_impl(ctx->peers[r], g->shards[r], binary ? 1 : 0, g->n_files, n_sets, set_offsets, chr, start, end, m,
                                      r == 0 ? out : nullptr, &barrier);
    });
}

// The count half of every single-device count: n device-resident queries of g's device (query i in set d_set_of[i]) into a
// zeroed [n_sets x n_files] matrix (scratch SC_MATRIX), copied to the host's out.  The caller holds ctx->mu.
static int32_t igd_count_to_host_locked(gtgpu_igd* g, bool binary, uint64_t n_sets, uint64_t n, const uint32_t* d_set,
                                        const uint32_t* d_chr, const uint32_t* d_start, const uint32_t* d_end, int32_t m, uint64_t* out) {
    gtgpu_ctx* ctx = g->ctx;
    cudaStream_t st = ctx->stream;
    uint64_t* d_out;
    const uint64_t cells = n_sets * g->n_files;
    GT_TRY(ctx->scratch_get(SC_MATRIX, cells * 8, (void**)&d_out));
    GT_CUDA(cudaMemsetAsync(d_out, 0, std::max<uint64_t>(cells * 8, 8), st));
    GT_TRY(igd_count_dev_locked(g, binary, n, d_set, d_chr, d_start, d_end, m, d_out));
    if (cells) GT_CUDA(cudaMemcpyAsync(out, d_out, cells * 8, cudaMemcpyDeviceToHost, st));
    GT_CUDA(cudaStreamSynchronize(st));
    return GTGPU_OK;
}

int32_t igd_count_host(gtgpu_igd* g, bool binary, uint64_t n_sets, const uint64_t* set_offsets, const uint32_t* chr,
                       const uint32_t* start, const uint32_t* end, int32_t m, uint64_t* out) {
    if (!g || !set_offsets || !out) return fail(GTGPU_ERR_INVALID, "igd count: null argument");
    if (!g->shards.empty()) return igd_count_group(g, binary, n_sets, set_offsets, chr, start, end, m, out);
    uint64_t n = set_offsets[n_sets];
    if (n && (!chr || !start || !end)) return fail(GTGPU_ERR_INVALID, "igd count: null query arrays");
    for (uint64_t s = 0; s < n_sets; ++s)
        if (set_offsets[s] > set_offsets[s + 1]) return fail(GTGPU_ERR_INVALID, "igd count: set_offsets not monotone");
    gtgpu_ctx* ctx = g->ctx;
    std::lock_guard<std::mutex> lk(ctx->mu);
    GT_CUDA(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    // the queries to the device
    uint32_t *d_chr, *d_start, *d_end, *d_set;
    uint64_t* d_so;
    GT_TRY(ctx->scratch_get(SC_CHR, n * 4, (void**)&d_chr));
    GT_TRY(ctx->scratch_get(SC_START, n * 4, (void**)&d_start));
    GT_TRY(ctx->scratch_get(SC_END, n * 4, (void**)&d_end));
    GT_TRY(ctx->scratch_get(SC_SET_ID, n * 4, (void**)&d_set));
    GT_TRY(ctx->scratch_get(SC_FILE_OFFS, (n_sets + 1) * 8, (void**)&d_so));
    if (n) {
        GT_CUDA(cudaMemcpyAsync(d_chr, chr, n * 4, cudaMemcpyHostToDevice, st));
        GT_CUDA(cudaMemcpyAsync(d_start, start, n * 4, cudaMemcpyHostToDevice, st));
        GT_CUDA(cudaMemcpyAsync(d_end, end, n * 4, cudaMemcpyHostToDevice, st));
    }
    GT_CUDA(cudaMemcpyAsync(d_so, set_offsets, (n_sets + 1) * 8, cudaMemcpyHostToDevice, st));
    if (n_sets && n) GT_TRY(launch_fill_set_ids(ctx, n_sets, d_so, d_set));
    return igd_count_to_host_locked(g, binary, n_sets, n, d_set, d_chr, d_start, d_end, m, out);
}

}  // namespace

extern "C" int32_t gtgpu_igd_count_set_overlaps(gtgpu_igd* igd, uint64_t n_sets, const uint64_t* set_offsets,
                                                const uint32_t* chr, const uint32_t* start, const uint32_t* end,
                                                int32_t min_overlap, uint64_t* out) try {
    return igd_count_host(igd, false, n_sets, set_offsets, chr, start, end, min_overlap, out);
} GT_CATCH

extern "C" int32_t gtgpu_igd_count_region_hits(gtgpu_igd* igd, uint64_t n_sets, const uint64_t* set_offsets,
                                               const uint32_t* chr, const uint32_t* start, const uint32_t* end,
                                               int32_t min_overlap, uint64_t* out) try {
    return igd_count_host(igd, true, n_sets, set_offsets, chr, start, end, min_overlap, out);
} GT_CATCH

extern "C" int32_t gtgpu_igd_count_dev(gtgpu_igd* igd, int32_t binary, uint64_t n, const uint32_t* d_set_of,
                                       const uint32_t* d_chr, const uint32_t* d_start, const uint32_t* d_end,
                                       int32_t min_overlap, uint64_t* d_out) try {
    if (!igd || (n && (!d_set_of || !d_chr || !d_start || !d_end || !d_out)))
        return fail(GTGPU_ERR_INVALID, "igd_count_dev: null argument");
    if (!igd->shards.empty())
        return fail(GTGPU_ERR_UNSUPPORTED, "igd_count_dev: device pointers belong to one device; a multi-device igd takes host arrays");
    std::lock_guard<std::mutex> lk(igd->ctx->mu);
    GT_CUDA(cudaSetDevice(igd->ctx->device));
    return igd_count_dev_locked(igd, binary != 0, n, d_set_of, d_chr, d_start, d_end, min_overlap, d_out);
} GT_CATCH

// ---- query sets from their BED files' text, parsed on the device (parse_bed_queries_locked) ---------------------------------
// The parsed query sets against g.  One device counts the columns where the parse left them; a group runs its sharded count
// with them as query arrays (each device pulls them from the first one) and gathers the shards' columns.
static int32_t igd_count_parsed(gtgpu_igd* g, bool binary, uint64_t n_sets, const BedFilesRecords& r, int32_t m, uint64_t* out,
                                uint64_t* out_set_regions) {
    gtgpu_ctx* ctx = g->ctx;
    if (!g->shards.empty()) {
        const int32_t s = igd_count_group(g, binary, n_sets, r.file_offsets.data(), r.chr.u32(), r.start.u32(), r.end.u32(), m, out);
        GT_CUDA(cudaSetDevice(ctx->device));  // the parsed records are freed on their device
        GT_TRY(s);
    } else {
        std::lock_guard<std::mutex> lk(ctx->mu);
        GT_CUDA(cudaSetDevice(ctx->device));
        GT_TRY(igd_count_to_host_locked(g, binary, n_sets, r.n, r.file.u32(), r.chr.u32(), r.start.u32(), r.end.u32(), m, out));
    }
    for (uint64_t s = 0; s < n_sets; ++s) out_set_regions[s] = r.file_offsets[s + 1] - r.file_offsets[s];
    return GTGPU_OK;
}

static int32_t igd_count_bed_check(const char* who, gtgpu_igd* igd, uint64_t n_sets, uint32_t n_names, const char* names,
                                   const uint32_t* name_offsets, int32_t min_overlap, uint64_t* out, uint64_t* out_set_regions) {
    if (!igd || !out || !out_set_regions || (n_names && (!names || !name_offsets)))
        return fail(GTGPU_ERR_INVALID, std::string(who) + ": null argument");
    if (n_sets >= 0xFFFFFFFFull) return fail(GTGPU_ERR_UNSUPPORTED, std::string(who) + ": too many sets");
    if (min_overlap < 1)
        return fail(GTGPU_ERR_UNSUPPORTED, std::string(who) + ": min_overlap < 1 depends on the reference's tile layout and is not supported");
    return GTGPU_OK;
}

extern "C" int32_t gtgpu_igd_count_bed(gtgpu_igd* igd, int32_t binary, uint64_t n_sets, const char* text, const uint64_t* file_offsets,
                                       uint32_t n_names, const char* names, const uint32_t* name_offsets, int32_t min_overlap,
                                       uint64_t* out, uint64_t* out_set_regions) try {
    GT_TRY(igd_count_bed_check("igd_count_bed", igd, n_sets, n_names, names, name_offsets, min_overlap, out, out_set_regions));
    if (!file_offsets) return fail(GTGPU_ERR_INVALID, "igd_count_bed: null argument");
    if (file_offsets[0] != 0) return fail(GTGPU_ERR_INVALID, "igd_count_bed: file_offsets[0] must be 0");
    for (uint64_t s = 0; s < n_sets; ++s)
        if (file_offsets[s] > file_offsets[s + 1]) return fail(GTGPU_ERR_INVALID, "igd_count_bed: file_offsets not monotone");
    if (file_offsets[n_sets] && !text) return fail(GTGPU_ERR_INVALID, "igd_count_bed: null text");
    if (n_sets == 0) return GTGPU_OK;
    gtgpu_ctx* ctx = igd->ctx;
    BedFilesRecords r;
    {
        std::lock_guard<std::mutex> lk(ctx->mu);
        GT_CUDA(cudaSetDevice(ctx->device));
        NameTable nt;
        GT_TRY(parse_bed_queries_locked(ctx, text, nullptr, n_sets, file_offsets, n_names, names, name_offsets, false, "igd_count_bed",
                                        &r, &nt));
    }
    return igd_count_parsed(igd, binary != 0, n_sets, r, min_overlap, out, out_set_regions);
} GT_CATCH

extern "C" int32_t gtgpu_igd_count_bed_gz(gtgpu_igd* igd, int32_t binary, uint64_t n_sets, const uint64_t* file_members,
                                          uint64_t n_members, const uint8_t* gz, const uint64_t* member_offsets, uint32_t n_names,
                                          const char* names, const uint32_t* name_offsets, int32_t min_overlap, uint64_t* out,
                                          uint64_t* out_set_regions) try {
    GT_TRY(igd_count_bed_check("igd_count_bed_gz", igd, n_sets, n_names, names, name_offsets, min_overlap, out, out_set_regions));
    if (!file_members) return fail(GTGPU_ERR_INVALID, "igd_count_bed_gz: null argument");
    GT_TRY(check_members(n_members, gz, member_offsets, "igd_count_bed_gz"));
    if (file_members[0] != 0 || file_members[n_sets] != n_members)
        return fail(GTGPU_ERR_INVALID, "igd_count_bed_gz: file_members must run from 0 to n_members");
    for (uint64_t s = 0; s < n_sets; ++s)
        if (file_members[s] > file_members[s + 1]) return fail(GTGPU_ERR_INVALID, "igd_count_bed_gz: file_members not monotone");
    if (n_sets == 0) return GTGPU_OK;
    gtgpu_ctx* ctx = igd->ctx;
    BedFilesRecords r;
    {
        std::lock_guard<std::mutex> lk(ctx->mu);
        GT_CUDA(cudaSetDevice(ctx->device));
        uint8_t* d_text = nullptr;
        uint64_t n_text = 0;
        std::vector<uint64_t> text_offsets(n_members + 1), fo(n_sets + 1);
        GT_TRY(inflate_whole_locked(ctx, n_members, gz, member_offsets, "igd_count_bed_gz", &d_text, &n_text, text_offsets.data()));
        for (uint64_t s = 0; s <= n_sets; ++s) fo[s] = text_offsets[file_members[s]];
        NameTable nt;
        GT_TRY(parse_bed_queries_locked(ctx, nullptr, (const char*)d_text, n_sets, fo.data(), n_names, names, name_offsets, false,
                                        "igd_count_bed_gz", &r, &nt));
    }
    return igd_count_parsed(igd, binary != 0, n_sets, r, min_overlap, out, out_set_regions);
} GT_CATCH

// ---- .igd bytes of a database, written from the device -----------------------------------------------------------------------
// Igd::save (igd.rs:418-486) after from_named_region_sets: a kept record sits in every 16 384-bp tile from start / nbp to
// (end - 1) / nbp of its contig, a tile holds its records stable-sorted by start with ties in (file, insertion) order, and the
// contigs come in the order Igd::add created them.  The pooled order (chromosome, start, file, insertion) filtered to one tile
// is that tile's order, so the records are expanded to one entry per tile they reach and sorted stably by (contig rank, tile).
namespace gtgpu {

constexpr int32_t IGD_NBP = 16384;  // igd.rs:14

// tiles[k] = the tiles record k reaches; tiles[n] = 0 closes the scan
__global__ void igd_tile_counts_kernel(uint64_t n, const int32_t* __restrict__ start, const int32_t* __restrict__ end,
                                       unsigned long long* __restrict__ tiles) {
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t k = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; k <= n; k += stride)
        tiles[k] = k < n ? (unsigned long long)((end[k] - 1) / IGD_NBP - start[k] / IGD_NBP + 1) : 0ull;
}

// one (global tile, record) pair per tile entry at the record's scanned offset; global tile = its contig's first tile + tile
__global__ void igd_expand_tiles_kernel(uint64_t n, const int32_t* __restrict__ start, const int32_t* __restrict__ end,
                                        const uint32_t* __restrict__ chr, const uint32_t* __restrict__ tile_base,
                                        const unsigned long long* __restrict__ offset, uint32_t* __restrict__ key,
                                        uint32_t* __restrict__ rec) {
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t k = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; k < n; k += stride) {
        const int32_t t0 = start[k] / IGD_NBP, t1 = (end[k] - 1) / IGD_NBP;
        const uint32_t b = tile_base[chr[k]] + (uint32_t)t0;
        const uint64_t o = offset[k];
        for (int32_t t = 0; t <= t1 - t0; ++t) {
            key[o + t] = b + (uint32_t)t;
            rec[o + t] = (uint32_t)k;
        }
    }
}

// entry j of the sorted order as the file's 16-byte record (file_idx, start, end, value = 0), one 16-byte store
__global__ void igd_format_records_kernel(uint64_t n, const uint32_t* __restrict__ perm, const uint32_t* __restrict__ rec,
                                          const uint32_t* __restrict__ file, const int32_t* __restrict__ start,
                                          const int32_t* __restrict__ end, int4* __restrict__ out) {
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; j < n; j += stride) {
        const uint32_t k = rec[perm[j]];
        out[j] = make_int4((int32_t)file[k], start[k], end[k], 0);
    }
}

__global__ void igd_add_u32_kernel(uint64_t n, uint32_t* __restrict__ v, uint32_t add) {
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t k = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; k < n; k += stride) v[k] += add;
}

}  // namespace gtgpu

// The records of a group igd on ctx's device in pooled order: every shard's arrays copied over (cudaMemcpyAsync, any device),
// file indexes rebased by the shard's first file, then stably sorted by (chromosome, start) as igd_build_dev step 1 does; shard
// order is file order, so ties keep (file, insertion).  The caller holds ctx->group_mu and ctx->mu.
static int32_t igd_gather_shards(gtgpu_igd* g, TempPool& tp, int32_t** out_start, int32_t** out_end, uint32_t** out_file,
                                 uint32_t** out_chr) {
    gtgpu_ctx* ctx = g->ctx;
    cudaStream_t st = ctx->stream;
    const uint64_t n = g->n_records;
    const uint32_t n_chroms = g->n_chroms;
    uint32_t *c_start, *c_end, *c_file, *c_chr;
    uint64_t* d_off64;
    GT_TRY(tp.get(n, &c_start));
    GT_TRY(tp.get(n, &c_end));
    GT_TRY(tp.get(n, &c_file));
    GT_TRY(tp.get(n, &c_chr));
    GT_TRY(tp.get(n, (uint32_t**)out_start));
    GT_TRY(tp.get(n, (uint32_t**)out_end));
    GT_TRY(tp.get(n, out_file));
    GT_TRY(tp.get(n, out_chr));
    GT_TRY(tp.get((uint64_t)n_chroms + 1, &d_off64));
    std::vector<uint64_t> off64(n_chroms + 1);
    uint64_t base = 0;
    for (gtgpu_igd* sh : g->shards) {
        const uint64_t m = sh->n_records;
        if (m == 0) continue;
        GT_CUDA(cudaMemcpyAsync(c_start + base, sh->d_start, m * 4, cudaMemcpyDefault, st));
        GT_CUDA(cudaMemcpyAsync(c_end + base, sh->d_end, m * 4, cudaMemcpyDefault, st));
        GT_CUDA(cudaMemcpyAsync(c_file + base, sh->d_file, m * 4, cudaMemcpyDefault, st));
        igd_add_u32_kernel<<<grid_for(ctx, m), 256, 0, st>>>(m, c_file + base, (uint32_t)sh->file0);
        for (uint32_t c = 0; c <= n_chroms; ++c) off64[c] = base + sh->h_off[c];
        GT_CUDA(cudaMemcpyAsync(d_off64, off64.data(), off64.size() * 8, cudaMemcpyHostToDevice, st));
        GT_TRY(launch_fill_set_ids(ctx, n_chroms, d_off64, c_chr));
        ctx->launches++;
        GT_CUDA(cudaGetLastError());
        GT_CUDA(cudaStreamSynchronize(st));  // off64 is reused for the next shard
        base += m;
    }
    if (n == 0) return GTGPU_OK;
    PermSorter pooled;
    GT_TRY(pooled.init(ctx, n));
    GT_TRY(pooled.pass(c_start, 0));
    GT_TRY(pooled.pass(c_chr, bits_for_value(n_chroms)));
    GT_TRY(launch_gather_u32(ctx, n, c_start, pooled.perm, (uint32_t*)*out_start));
    GT_TRY(launch_gather_u32(ctx, n, c_end, pooled.perm, (uint32_t*)*out_end));
    GT_TRY(launch_gather_u32(ctx, n, c_file, pooled.perm, *out_file));
    GT_TRY(launch_gather_u32(ctx, n, c_chr, pooled.perm, *out_chr));
    GT_CUDA(cudaStreamSynchronize(st));
    return GTGPU_OK;
}

// n kept records in pooled order on ctx's device -> the record payload of the file (16 bytes per tile entry) at buf + header,
// where the header is written from the tile counts.  tile_base[c]: the first global tile of chromosome c's contig; the contigs'
// tiles are numbered in file order, n_tiles in all.  The caller holds ctx->mu.
static int32_t igd_write_tiles_locked(gtgpu_ctx* ctx, TempPool& tp, uint64_t n, const int32_t* d_start, const int32_t* d_end,
                                      const uint32_t* d_file, const uint32_t* d_chr, const std::vector<uint32_t>& tile_base,
                                      uint64_t n_tiles, uint64_t header_bytes, BufPtr* out_buf, std::vector<uint32_t>* tile_off) {
    cudaStream_t st = ctx->stream;
    unsigned long long *d_tiles, *d_toff;
    char* d_scan_tmp;
    GT_TRY(tp.get(n + 1, &d_tiles));
    GT_TRY(tp.get(n + 1, &d_toff));
    GT_TRY(tp.get(exclusive_scan_temp_bytes(n + 1, 8), &d_scan_tmp));
    igd_tile_counts_kernel<<<grid_for(ctx, n + 1), 256, 0, st>>>(n, d_start, d_end, d_tiles);
    ctx->launches++;
    GT_CUDA(cudaGetLastError());
    GT_TRY(exclusive_scan<unsigned long long>(ctx, d_tiles, d_toff, n + 1, d_scan_tmp));
    uint64_t entries = 0;
    GT_CUDA(cudaMemcpyAsync(&entries, d_toff + n, 8, cudaMemcpyDeviceToHost, st));
    GT_CUDA(cudaStreamSynchronize(st));
    if (entries >= 0xFFFFFFFFull)
        return fail(GTGPU_ERR_UNSUPPORTED, "igd_serialize: " + std::to_string(entries) + " tile entries (at most 2^32 - 2)");
    uint32_t *d_key, *d_rec, *d_tile_base, *d_tile_off;
    int4* d_payload;
    GT_TRY(tp.get(entries, &d_key));
    GT_TRY(tp.get(entries, &d_rec));
    GT_TRY(tp.get(tile_base.size(), &d_tile_base));
    GT_TRY(tp.get(n_tiles + 1, &d_tile_off));
    GT_TRY(tp.get(entries, &d_payload));
    if (!tile_base.empty())
        GT_CUDA(cudaMemcpyAsync(d_tile_base, tile_base.data(), tile_base.size() * 4, cudaMemcpyHostToDevice, st));
    BufPtr buf;
    GT_TRY(buf_new(ctx, header_bytes + entries * 16, 1, &buf));
    tile_off->assign(n_tiles + 1, 0);
    if (entries) {
        igd_expand_tiles_kernel<<<grid_for(ctx, n), 256, 0, st>>>(n, d_start, d_end, d_chr, d_tile_base, d_toff, d_key, d_rec);
        ctx->launches++;
        GT_CUDA(cudaGetLastError());
        PermSorter by_tile;
        GT_TRY(by_tile.init(ctx, entries));
        GT_TRY(by_tile.pass(d_key, bits_for_value(n_tiles - 1)));
        GT_TRY(launch_key_offsets(ctx, entries, by_tile.key, (uint32_t)n_tiles, d_tile_off));
        igd_format_records_kernel<<<grid_for(ctx, entries), 256, 0, st>>>(entries, by_tile.perm, d_rec, d_file, d_start, d_end,
                                                                           d_payload);
        ctx->launches++;
        GT_CUDA(cudaGetLastError());
        GT_CUDA(cudaMemcpyAsync(tile_off->data(), d_tile_off, (n_tiles + 1) * 4, cudaMemcpyDeviceToHost, st));
        GT_CUDA(cudaMemcpyAsync((char*)buf->block.ptr + header_bytes, d_payload, entries * 16, cudaMemcpyDeviceToHost, st));
        GT_CUDA(cudaStreamSynchronize(st));  // by_tile is freed when it leaves
    }
    *out_buf = std::move(buf);
    return GTGPU_OK;
}

extern "C" int32_t gtgpu_igd_serialize(gtgpu_igd* g, uint32_t n_names, const char* names, const uint32_t* name_offsets,
                                       gtgpu_buf** out_igd_bytes, uint64_t* out_file_regions, uint64_t* out_file_width_sums) try {
    if (!g || !out_igd_bytes || (g->n_files && (!out_file_regions || !out_file_width_sums)) || (n_names && (!names || !name_offsets)))
        return fail(GTGPU_ERR_INVALID, "igd_serialize: null argument");
    if (n_names != g->n_chroms)
        return fail(GTGPU_ERR_INVALID, "igd_serialize: " + std::to_string(n_names) + " names for " + std::to_string(g->n_chroms) +
                                           " chromosomes");
    for (uint32_t c = 0; c < n_names; ++c)
        if (name_offsets[c] > name_offsets[c + 1]) return fail(GTGPU_ERR_INVALID, "igd_serialize: name_offsets not monotone");
    gtgpu_ctx* ctx = g->ctx;
    const std::vector<gtgpu_igd*> parts = g->shards.empty() ? std::vector<gtgpu_igd*>{g} : g->shards;
    const uint32_t n_chroms = g->n_chroms;
    // the .tsv numbers, and per chromosome its rank key and largest end over the parts
    std::vector<uint64_t> first(n_chroms, UINT64_MAX);
    std::vector<uint32_t> max_end(n_chroms, 0);
    for (const gtgpu_igd* p : parts) {
        std::copy(p->h_file_regions.begin(), p->h_file_regions.end(), out_file_regions + p->file0);
        std::copy(p->h_file_widths.begin(), p->h_file_widths.end(), out_file_width_sums + p->file0);
        const uint64_t rebase = g->contig_by_file ? p->file0 : p->rec0;
        for (uint32_t c = 0; c < n_chroms; ++c) {
            if (p->h_off[c + 1] == p->h_off[c]) continue;
            first[c] = std::min<uint64_t>(first[c], p->h_first[c] + rebase);
            max_end[c] = std::max(max_end[c], p->h_max_end[c]);
        }
    }
    // contigs in creation order: by first kept input index (distinct), or for BED files by (first file, name bytes)
    std::vector<uint32_t> order;
    for (uint32_t c = 0; c < n_chroms; ++c)
        if (first[c] != UINT64_MAX) order.push_back(c);
    auto name = [&](uint32_t c) { return std::string(names + name_offsets[c], names + name_offsets[c + 1]); };
    std::sort(order.begin(), order.end(), [&](uint32_t a, uint32_t b) {
        if (first[a] != first[b]) return first[a] < first[b];
        return name(a).compare(name(b)) < 0;
    });
    std::vector<uint32_t> tile_base(n_chroms, 0), contig_tiles(order.size());
    uint64_t n_tiles = 0;
    for (size_t i = 0; i < order.size(); ++i) {
        contig_tiles[i] = (max_end[order[i]] - 1) / IGD_NBP + 1;
        tile_base[order[i]] = (uint32_t)n_tiles;
        n_tiles += contig_tiles[i];
        if (n_tiles >= 0x7FFFFFFFull) return fail(GTGPU_ERR_UNSUPPORTED, "igd_serialize: 2^31 - 1 tiles or more");
    }
    const uint64_t n_ctg = order.size(), header_bytes = 12 + 4 * n_ctg + 4 * n_tiles + 40 * n_ctg;

    std::unique_lock<std::mutex> glk;
    if (!g->shards.empty()) glk = std::unique_lock<std::mutex>(ctx->group_mu);
    std::lock_guard<std::mutex> lk(ctx->mu);
    GT_CUDA(cudaSetDevice(ctx->device));
    TempPool tp;
    const uint64_t n = g->n_records;
    int32_t *d_start = g->d_start, *d_end = g->d_end;
    uint32_t *d_file = g->d_file, *d_chr;
    if (g->shards.empty()) {
        uint64_t* d_off64;
        GT_TRY(tp.get(n, &d_chr));
        GT_TRY(tp.get((uint64_t)n_chroms + 1, &d_off64));
        const std::vector<uint64_t> off64(g->h_off.begin(), g->h_off.end());
        GT_CUDA(cudaMemcpyAsync(d_off64, off64.data(), off64.size() * 8, cudaMemcpyHostToDevice, ctx->stream));
        if (n) GT_TRY(launch_fill_set_ids(ctx, n_chroms, d_off64, d_chr));
        GT_CUDA(cudaStreamSynchronize(ctx->stream));  // off64 is pageable
    } else {
        GT_TRY(igd_gather_shards(g, tp, &d_start, &d_end, &d_file, &d_chr));
    }
    BufPtr buf;
    std::vector<uint32_t> tile_off;
    GT_TRY(igd_write_tiles_locked(ctx, tp, n, d_start, d_end, d_file, d_chr, tile_base, n_tiles, header_bytes, &buf, &tile_off));

    // the header: nbp, gType 1 (16-byte records), nCtg; nTile per contig; nCnt per tile; 40-byte NUL-padded names (igd.rs:418-486)
    char* h = (char*)buf->block.ptr;
    auto put = [&](int32_t v) {
        memcpy(h, &v, 4);
        h += 4;
    };
    put(IGD_NBP);
    put(1);
    put((int32_t)n_ctg);
    for (uint32_t t : contig_tiles) put((int32_t)t);
    for (uint64_t t = 0; t < n_tiles; ++t) put((int32_t)(tile_off[t + 1] - tile_off[t]));
    for (uint32_t c : order) {
        const uint32_t len = std::min<uint32_t>(name_offsets[c + 1] - name_offsets[c], 40);
        memset(h, 0, 40);
        memcpy(h, names + name_offsets[c], len);
        h += 40;
    }
    *out_igd_bytes = buf.release();
    return GTGPU_OK;
} GT_CATCH
