// sort.cu — hand-written device primitives: exclusive scan and a stable LSD radix sort of (key, value) pairs.
//
// Used by the barcode group-by of fragment tokenization (fragments.cu).  Both are plain multi-kernel designs (no
// single-pass tricks): they run once per call over arrays that are small next to the fused find kernel's traffic.
//
//   exclusive_scan<T>:  reduce per 2 048-element tile -> scan of the tile sums by one block -> per-tile rescan + offset.
//   radix_sort_pairs:   8 (or 9, when that saves a pass) bits per pass; per pass  (1) per-tile digit histograms, stored digit-major,
//                       (2) exclusive scan of that table = global start of every (digit, tile) bucket,
//                       (3) scatter: each warp owns 512 consecutive elements, ranks them round by round with
//                           __match_any_sync, so equal digits keep their input order (stable).
#include <algorithm>

#include "common.cuh"

namespace gtgpu {

constexpr int SCAN_THREADS = 256;
constexpr int SCAN_ITEMS = 8;
constexpr int SCAN_TILE = SCAN_THREADS * SCAN_ITEMS;

template <typename T>
__device__ __forceinline__ T block_exclusive_scan(T v, T* s_warp, T& total) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    T incl = v;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        T t = __shfl_up_sync(0xFFFFFFFFu, incl, d);
        if (lane >= d) incl += t;
    }
    if (lane == 31) s_warp[warp] = incl;
    __syncthreads();
    T warp_excl = 0, tot = 0;
#pragma unroll
    for (int w = 0; w < SCAN_THREADS / 32; ++w) {
        const T t = s_warp[w];
        if (w < warp) warp_excl += t;
        tot += t;
    }
    __syncthreads();
    total = tot;
    return warp_excl + incl - v;
}

template <typename T>
__global__ void __launch_bounds__(SCAN_THREADS) scan_reduce_kernel(const T* __restrict__ in, T* __restrict__ tile_sums, uint64_t n) {
    __shared__ T s_warp[SCAN_THREADS / 32];
    const uint64_t base = (uint64_t)blockIdx.x * SCAN_TILE;
    T sum = 0;
#pragma unroll
    for (int k = 0; k < SCAN_ITEMS; ++k) {
        const uint64_t i = base + (uint64_t)k * SCAN_THREADS + threadIdx.x;
        if (i < n) sum += in[i];
    }
    T total;
    block_exclusive_scan<T>(sum, s_warp, total);
    if (threadIdx.x == 0) tile_sums[blockIdx.x] = total;
}

template <typename T>
__global__ void __launch_bounds__(SCAN_THREADS) scan_spine_kernel(T* __restrict__ tile_sums, uint64_t n_tiles) {
    __shared__ T s_warp[SCAN_THREADS / 32];
    T carry = 0;
    for (uint64_t base = 0; base < n_tiles; base += SCAN_THREADS) {
        const uint64_t i = base + threadIdx.x;
        const T v = i < n_tiles ? tile_sums[i] : 0;
        T total;
        const T excl = block_exclusive_scan<T>(v, s_warp, total);
        if (i < n_tiles) tile_sums[i] = carry + excl;
        carry += total;
    }
}

template <typename T>
__global__ void __launch_bounds__(SCAN_THREADS) scan_down_kernel(const T* __restrict__ in, T* __restrict__ out,
                                                                  const T* __restrict__ tile_offsets, uint64_t n) {
    __shared__ T s_warp[SCAN_THREADS / 32];
    const uint64_t base = (uint64_t)blockIdx.x * SCAN_TILE + (uint64_t)threadIdx.x * SCAN_ITEMS;  // blocked: 8 consecutive
    T v[SCAN_ITEMS];
    T sum = 0;
#pragma unroll
    for (int k = 0; k < SCAN_ITEMS; ++k) {
        v[k] = base + k < n ? in[base + k] : 0;
        sum += v[k];
    }
    T total;
    T run = tile_offsets[blockIdx.x] + block_exclusive_scan<T>(sum, s_warp, total);
#pragma unroll
    for (int k = 0; k < SCAN_ITEMS; ++k) {
        if (base + k < n) out[base + k] = run;
        run += v[k];
    }
}

size_t exclusive_scan_temp_bytes(uint64_t n, size_t elem) { return (size_t)((n + SCAN_TILE - 1) / SCAN_TILE + 1) * elem; }

template <typename T>
int32_t exclusive_scan(gtgpu_ctx* ctx, const T* d_in, T* d_out, uint64_t n, void* d_temp) {
    if (n == 0) return GTGPU_OK;
    const uint64_t tiles = (n + SCAN_TILE - 1) / SCAN_TILE;
    if (tiles > 0x7FFFFFFFull) return fail(GTGPU_ERR_UNSUPPORTED, "exclusive_scan: input too large");
    T* sums = reinterpret_cast<T*>(d_temp);
    scan_reduce_kernel<T><<<(unsigned)tiles, SCAN_THREADS, 0, ctx->stream>>>(d_in, sums, n);
    scan_spine_kernel<T><<<1, SCAN_THREADS, 0, ctx->stream>>>(sums, tiles);
    scan_down_kernel<T><<<(unsigned)tiles, SCAN_THREADS, 0, ctx->stream>>>(d_in, d_out, sums, n);
    ctx->launches += 3;
    GT_CUDA(cudaGetLastError());
    return GTGPU_OK;
}
template int32_t exclusive_scan<uint32_t>(gtgpu_ctx*, const uint32_t*, uint32_t*, uint64_t, void*);
template int32_t exclusive_scan<unsigned long long>(gtgpu_ctx*, const unsigned long long*, unsigned long long*, uint64_t, void*);

// ---- inclusive running maximum (64-bit) ---------------------------------------------------------------------------------
// Same three-kernel shape as exclusive_scan with max as the operator.  The index builders use it for segmented running
// maxima: with the segment number in the high word and the value in the low word, a later segment always wins, so the
// low word of the scan is the running maximum inside the element's own segment.
__device__ __forceinline__ unsigned long long block_inclusive_max(unsigned long long v, unsigned long long* s_warp,
                                                                  unsigned long long& total) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    unsigned long long incl = v;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const unsigned long long t = __shfl_up_sync(0xFFFFFFFFu, incl, d);
        if (lane >= d) incl = max(incl, t);
    }
    if (lane == 31) s_warp[warp] = incl;
    __syncthreads();
    unsigned long long before = 0, tot = 0;
#pragma unroll
    for (int w = 0; w < SCAN_THREADS / 32; ++w) {
        const unsigned long long t = s_warp[w];
        if (w < warp) before = max(before, t);
        tot = max(tot, t);
    }
    __syncthreads();
    total = tot;
    return max(before, incl);
}

__global__ void __launch_bounds__(SCAN_THREADS) max_reduce_kernel(const unsigned long long* __restrict__ in,
                                                                  unsigned long long* __restrict__ tile_max, uint64_t n) {
    __shared__ unsigned long long s_warp[SCAN_THREADS / 32];
    const uint64_t base = (uint64_t)blockIdx.x * SCAN_TILE;
    unsigned long long m = 0;
#pragma unroll
    for (int k = 0; k < SCAN_ITEMS; ++k) {
        const uint64_t i = base + (uint64_t)k * SCAN_THREADS + threadIdx.x;
        if (i < n) m = max(m, in[i]);
    }
    unsigned long long total;
    block_inclusive_max(m, s_warp, total);
    if (threadIdx.x == 0) tile_max[blockIdx.x] = total;
}

// tile_max[t] becomes the maximum over all tiles BEFORE t (0 for the first)
__global__ void __launch_bounds__(SCAN_THREADS) max_spine_kernel(unsigned long long* __restrict__ tile_max, uint64_t n_tiles) {
    __shared__ unsigned long long s_warp[SCAN_THREADS / 32];
    __shared__ unsigned long long s_prev[SCAN_THREADS];
    unsigned long long carry = 0;
    for (uint64_t base = 0; base < n_tiles; base += SCAN_THREADS) {
        const uint64_t i = base + threadIdx.x;
        const unsigned long long v = i < n_tiles ? tile_max[i] : 0;
        unsigned long long total;
        const unsigned long long incl = block_inclusive_max(v, s_warp, total);
        s_prev[threadIdx.x] = incl;
        __syncthreads();
        const unsigned long long excl = threadIdx.x ? s_prev[threadIdx.x - 1] : 0;
        if (i < n_tiles) tile_max[i] = max(carry, excl);
        carry = max(carry, total);
        __syncthreads();
    }
}

// in and out may be the same array (every thread reads its own eight elements before it writes them): no __restrict__
__global__ void __launch_bounds__(SCAN_THREADS) max_down_kernel(const unsigned long long* in, unsigned long long* out,
                                                                const unsigned long long* __restrict__ tile_before, uint64_t n) {
    __shared__ unsigned long long s_warp[SCAN_THREADS / 32];
    __shared__ unsigned long long s_prev[SCAN_THREADS];
    const uint64_t base = (uint64_t)blockIdx.x * SCAN_TILE + (uint64_t)threadIdx.x * SCAN_ITEMS;
    unsigned long long v[SCAN_ITEMS], m = 0;
#pragma unroll
    for (int k = 0; k < SCAN_ITEMS; ++k) {
        v[k] = base + k < n ? in[base + k] : 0;
        m = max(m, v[k]);
    }
    unsigned long long total;
    s_prev[threadIdx.x] = block_inclusive_max(m, s_warp, total);
    __syncthreads();
    unsigned long long run = max(tile_before[blockIdx.x], threadIdx.x ? s_prev[threadIdx.x - 1] : 0ull);
#pragma unroll
    for (int k = 0; k < SCAN_ITEMS; ++k) {
        run = max(run, v[k]);
        if (base + k < n) out[base + k] = run;
    }
}

// out[i] = max(in[0..i]); in and out may alias; d_temp needs exclusive_scan_temp_bytes(n, 8).
int32_t inclusive_max_scan_u64(gtgpu_ctx* ctx, const unsigned long long* d_in, unsigned long long* d_out, uint64_t n, void* d_temp) {
    if (n == 0) return GTGPU_OK;
    const uint64_t tiles = (n + SCAN_TILE - 1) / SCAN_TILE;
    if (tiles > 0x7FFFFFFFull) return fail(GTGPU_ERR_UNSUPPORTED, "inclusive_max_scan: input too large");
    unsigned long long* tm = reinterpret_cast<unsigned long long*>(d_temp);
    max_reduce_kernel<<<(unsigned)tiles, SCAN_THREADS, 0, ctx->stream>>>(d_in, tm, n);
    max_spine_kernel<<<1, SCAN_THREADS, 0, ctx->stream>>>(tm, tiles);
    max_down_kernel<<<(unsigned)tiles, SCAN_THREADS, 0, ctx->stream>>>(d_in, d_out, tm, n);
    ctx->launches += 3;
    GT_CUDA(cudaGetLastError());
    return GTGPU_OK;
}

// ---- radix sort -----------------------------------------------------------------------------------------------------------
// lanes with equal digits: one ballot per digit bit (C5: 26.3 ms per 1e9 fragments) or __match_any_sync (27.6 ms)
#ifndef GT_RS_BALLOT
#define GT_RS_BALLOT 1
#endif
constexpr int RS_HIST_THREADS = 512;

// Shape of the scatter kernel: threads per block, elements per lane ("rounds": the length of a warp's ranking chain), blocks
// per SM.  The tile (threads x rounds) is also the histogram kernel's tile.  Shared memory per block = 8 B per tile element +
// 2 B per (warp, digit) counter + 8 B per digit, so a shorter tile buys resident warps: the kernel is bound by the latency of
// its phases (load, rank, stage, write), not by a pipe, and what hides that latency is other blocks in other phases.
struct RsShape {
    int threads, rounds, min_blocks;
};
constexpr RsShape RS_SHAPES[] = {
    {512, 16, 2},   // 0: 8 192-element tile, 32 warps per SM — the default: 24.9 ms per 1e9 fragments on C5
    {512, 12, 3},   // 1: 6 144, 48 warps: 27.4 ms (shorter runs, a larger bucket table)
    {1024, 16, 1},  // 2: 16 384, 32 warps in one block: 27.9 ms (nothing overlaps the block's own phases)
};
// also measured (profiles/r02/c5_scatter_shape_sweep_*.jsonl): 512 x 8 x 4 blocks, 256 x 16 x 4 / 5, 256 x 12 x 6, 1 024 x 8 x 2,
// 1 024 x 20 x 1 — all slower than shape 0 — and a shared-memory table instead of the ballots (every lane writes its lane number
// at its digit and reads the slot back, only shared digits are then resolved by votes): 35 % fewer instructions, but the kernel is
// as busy in the shared-memory pipe as in the issue slots, and two more conflicted accesses per round made it 4 % slower
// (profiles/r02/c5_scatter_table_match_sweep.jsonl).
constexpr int RS_N_SHAPES = (int)(sizeof(RS_SHAPES) / sizeof(RS_SHAPES[0]));
#ifndef GT_RS_DEFAULT_SHAPE
#define GT_RS_DEFAULT_SHAPE 0
#endif

// run-time choice (GTGPU_RS_SHAPE, for sweeps; read at every call so that one process can compare shapes)
static int rs_shape_index() {
    const char* e = getenv("GTGPU_RS_SHAPE");
    if (e && *e) {
        const int v = atoi(e);
        if (v >= 0 && v < RS_N_SHAPES) return v;
    }
    return GT_RS_DEFAULT_SHAPE;
}

// DB = digit width of the pass: 8 bits, or 9 when that saves a whole pass (17-18 and 25-27 significant bits)
template <int DB, int TILE>
__global__ void __launch_bounds__(RS_HIST_THREADS) radix_hist_kernel(const uint32_t* __restrict__ keys, uint64_t n_cap,
                                                                     const uint64_t* __restrict__ d_n, int shift,
                                                                     uint32_t n_tiles, uint32_t* __restrict__ hist) {
    constexpr uint32_t ND = 1u << DB;
    constexpr int WARPS = RS_HIST_THREADS / 32;
    constexpr int ROUNDS = (TILE + RS_HIST_THREADS - 1) / RS_HIST_THREADS;
    const uint64_t n = d_n ? min((uint64_t)*d_n, n_cap) : n_cap;  // element count known on the device only (no host sync)
    // one histogram per warp pair (little contention; a warp's 32 lanes rarely share a digit), summed at the end
    __shared__ uint32_t s_hist[WARPS / 2][ND];
    for (uint32_t i = threadIdx.x; i < (WARPS / 2) * ND; i += RS_HIST_THREADS) (&s_hist[0][0])[i] = 0;
    __syncthreads();
    const uint64_t base = (uint64_t)blockIdx.x * TILE;
    const uint64_t lim = min(n, base + TILE);
    uint32_t* mine = s_hist[(threadIdx.x >> 5) >> 1];
    // all loads of a thread in flight before the first atomic (four at a time left the DRAM at a quarter of its rate)
    uint32_t key[ROUNDS];
#pragma unroll
    for (int k = 0; k < ROUNDS; ++k) {
        const uint64_t i = base + (uint64_t)k * RS_HIST_THREADS + threadIdx.x;
        key[k] = i < lim ? __ldcs(keys + i) : 0;
    }
#pragma unroll
    for (int k = 0; k < ROUNDS; ++k)
        if (base + (uint64_t)k * RS_HIST_THREADS + threadIdx.x < lim) atomicAdd(&mine[(key[k] >> shift) & (ND - 1)], 1u);
    __syncthreads();
    for (uint32_t d = threadIdx.x; d < ND; d += RS_HIST_THREADS) {
        uint32_t t = 0;
#pragma unroll
        for (int w = 0; w < WARPS / 2; ++w) t += s_hist[w][d];
        hist[(uint64_t)d * n_tiles + blockIdx.x] = t;  // digit-major: one scan orders everything
    }
}

// Scatter of one pass.  A block sorts its tile by digit in SHARED memory first (stable: per-warp ranks from the set of lanes
// with the same digit, round by round, warps in order), then writes the tile out digit by digit — a digit's elements of one
// tile go to consecutive addresses, so the global stores are coalesced runs instead of single words.  (The first version
// stored every element straight from its ranking round: 16 scattered 4-byte stores per lane and array, 9.8 ms per 2.5e8
// pairs; the second held the keys in registers and fetched the values in the middle of the kernel: 64 registers, two blocks
// per SM, two exposed load latencies per tile; see profiles/r02.)
//
// The tile arrives by cp.async at the very top — keys into the buffer that will hold the sorted VALUES, values into the buffer
// that will hold the sorted KEYS — and the kernel only waits for the keys before it ranks; the values land while it does.
// Ranking reads the keys back from shared memory round by round (conflict-free: a warp's round is 32 consecutive words), so
// the only per-element state in registers is the 16-bit rank (two per register).  The swap into sorted order lifts the
// values into registers, moves the keys buffer to buffer, then drops the values: ROUNDS registers at the peak instead of
// 3 x ROUNDS, which is what lets the shorter shapes keep three or four blocks on an SM without spilling.
__device__ __forceinline__ uint32_t rs_smem_addr(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void rs_cp_async16(void* s, const void* g) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(rs_smem_addr(s)), "l"(g) : "memory");
}
__device__ __forceinline__ void rs_cp_async4(void* s, const void* g) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(rs_smem_addr(s)), "l"(g) : "memory");
}
__device__ __forceinline__ void rs_cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void rs_cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// tile_n words from g to s: 16-byte copies when the source is aligned and the tile is full, single words otherwise
template <int THREADS, int TILE>
__device__ __forceinline__ void rs_stage_tile(uint32_t* s, const uint32_t* g, uint32_t tile_n, uint32_t tid) {
    if (tile_n == TILE && (reinterpret_cast<uintptr_t>(g) & 15) == 0) {
#pragma unroll
        for (uint32_t c = tid; c < TILE / 4; c += THREADS) rs_cp_async16(s + 4 * c, g + 4 * c);
    } else {
        for (uint32_t j = tid; j < tile_n; j += THREADS) rs_cp_async4(s + j, g + j);
    }
}

//
// MODE: what moves.  RS_PAIRS: (key, value) in, (key, value) out.  RS_PACK: (key, value) in, ONE word out —
// (key >> (shift + DB)) << aux | value: the key bits no later pass has sorted yet, next to the value.  RS_KEYS: one word in,
// word & aux out (to vals_out) — the last pass over such packed words sheds the key.  radix_group_values runs PACK then KEYS:
// 20 instead of 32 bytes of scatter traffic per element, and the second pass moves one array through shared memory, not two.
enum { RS_PAIRS = 0, RS_PACK = 1, RS_KEYS = 2 };

// peers &= the lanes whose digit agrees with mine in bit `bit`, in PTX — the plain C++
// (`peers &= (d & bit) ? bal : ~bal`) compiled to seven instructions per bit (shift, mask, compare, vote, test, select, combine;
// this form: one R2P for seven bits, then vote, select, combine),
// and the ten votes of a round with their arithmetic were 45 % of the kernel's instructions
__device__ __forceinline__ void rs_match_bit(uint32_t& peers, uint32_t d, uint32_t bit) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        ".reg .b32 t, bal;\n"
        "and.b32 t, %1, %2;\n"
        "setp.ne.u32 p, t, 0;\n"
        "vote.sync.ballot.b32 bal, p, 0xffffffff;\n"
        "selp.b32 t, 0, 0xffffffff, p;\n"
        "lop3.b32 %0, %0, bal, t, 0x60;\n"  // peers & (bal ^ t): bal where my bit is set, ~bal where it is not
        "}\n" : "+r"(peers) : "r"(d), "r"(bit));
}

// FULL: every element of the tile exists (all tiles but the last): no bounds tests, no predicates on the element accesses
template <int DB, int THREADS, int ROUNDS, int MODE, bool FULL>
__device__ __forceinline__ void rs_scatter_tile(const uint32_t* __restrict__ keys_in, const uint32_t* __restrict__ vals_in,
                                                uint64_t tile0, uint32_t tile_n, int shift, uint32_t n_tiles,
                                                const uint32_t* __restrict__ bucket_start, uint32_t* __restrict__ keys_out,
                                                uint32_t* __restrict__ vals_out, uint32_t aux, uint32_t* s_mem, uint32_t* s_wsum) {
    constexpr uint32_t ND = 1u << DB;
    constexpr int WARPS = THREADS / 32, TILE = THREADS * ROUNDS, WARP_TILE = 32 * ROUNDS;
    constexpr int DPT = (int)ND > THREADS ? (int)ND / THREADS : 1;  // digits per thread in phase 2
    uint32_t* s_key = s_mem;                                       // [TILE] the values as they arrive, then the keys sorted by digit
    uint32_t* s_val = s_mem + TILE;                                // [TILE] the keys as they arrive, then the values sorted by digit
    uint32_t* s_dbase = s_mem + 2 * TILE;                          // [ND] first slot of each digit in the sorted tile
    uint32_t* s_gbase = s_dbase + ND;                              // [ND] global position of the digit's first element minus s_dbase
    uint16_t* s_cnt = reinterpret_cast<uint16_t*>(s_gbase + ND);   // [WARPS][ND] per-warp digit counts (<= 32 x ROUNDS), then
                                                                   // the digit's elements in earlier warps (<= TILE < 65 536)
    const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
#define RS_OK(r) (FULL || wbase + 32 * (r) < tile_n)
    uint32_t* in_key = s_val;  // arrival buffers
    uint32_t* in_val = s_key;
    rs_stage_tile<THREADS, TILE>(in_key, keys_in + tile0, FULL ? TILE : tile_n, tid);
    rs_cp_async_commit();
    if (MODE != RS_KEYS) rs_stage_tile<THREADS, TILE>(in_val, vals_in + tile0, FULL ? TILE : tile_n, tid);
    rs_cp_async_commit();  // (an empty group when there are no values)
    // this tile's row of the bucket table (a gather: the table is digit-major), requested now, used after phase 2
    const bool has_digits = tid * DPT < ND;
    uint32_t gstart[DPT];
    if (has_digits) {
#pragma unroll
        for (int k = 0; k < DPT; ++k) gstart[k] = __ldg(bucket_start + (uint64_t)(tid * DPT + k) * n_tiles + blockIdx.x);
    }
    for (uint32_t i = tid; i < WARPS * ND / 2; i += THREADS) reinterpret_cast<uint32_t*>(s_cnt)[i] = 0;
    rs_cp_async_wait<1>();  // my pieces of the keys have landed ...
    __syncthreads();        // ... everyone's have, and the counters are zero
    // ---- 1. rank inside the warp, round by round (stable) ----------------------------------------------------------------
    const uint32_t wbase = warp * WARP_TILE + lane;
    uint32_t rank2[ROUNDS / 2];  // two 16-bit ranks per register
    uint16_t* my_cnt = s_cnt + warp * ND;
    // the matches do not depend on each other: issue them ahead of the counter rounds (a match per round in front of that
    // round's counter update left every warp waiting on its result: a third of the kernel's stall samples) ...
#pragma unroll
    for (int r = 0; r < ROUNDS; ++r) {
        const bool ok = RS_OK(r);
        const uint32_t d = ok ? (in_key[wbase + 32 * r] >> shift) & (ND - 1) : ND + lane;  // invalid lanes never match anyone
#if GT_RS_BALLOT
        uint32_t peers = FULL ? 0xFFFFFFFFu : __ballot_sync(0xFFFFFFFFu, ok);
#pragma unroll
        for (int b = 0; b < DB; ++b) rs_match_bit(peers, d, 1u << b);
        if (!ok) peers = 1u << lane;
#else
        const uint32_t peers = __match_any_sync(0xFFFFFFFFu, d);
#endif
        const uint32_t packed = __popc(peers & ((1u << lane) - 1)) | __popc(peers) << 8;  // lanes before me | group size
        if (r & 1) rank2[r >> 1] |= packed << 16;
        else rank2[r >> 1] = packed;
    }
    // ... then the per-warp digit counters advance round by round (stable)
#pragma unroll
    for (int r = 0; r < ROUNDS; ++r) {
        const bool ok = RS_OK(r);
        const uint32_t mine = (r & 1) ? rank2[r >> 1] >> 16 : rank2[r >> 1] & 0xFFFFu;
        const uint32_t d = ok ? (in_key[wbase + 32 * r] >> shift) & (ND - 1) : 0, before = mine & 0xFFu, group = mine >> 8;
        uint32_t prev = 0;
        if (ok) prev = my_cnt[d];
        __syncwarp();
        if (ok && before == 0) my_cnt[d] = (uint16_t)(prev + group);
        __syncwarp();
        if (r & 1) rank2[r >> 1] = (rank2[r >> 1] & 0xFFFFu) | (prev + before) << 16;
        else rank2[r >> 1] = (rank2[r >> 1] & 0xFFFF0000u) | (prev + before);
    }
    __syncthreads();
    // ---- 2. digit totals -> first slot of every digit, and of every (warp, digit) ------------------------------------------
    uint32_t tot = 0, sub[DPT];  // thread t: digits [t * DPT, (t + 1) * DPT)
    if (has_digits) {
#pragma unroll
        for (int k = 0; k < DPT; ++k) {
            const uint32_t d = tid * DPT + k;
            uint32_t run = 0;
#pragma unroll
            for (int w = 0; w < WARPS; ++w) {
                const uint32_t c = s_cnt[w * ND + d];
                s_cnt[w * ND + d] = (uint16_t)run;  // elements of this digit in earlier warps
                run += c;
            }
            sub[k] = run;
            tot += run;
        }
    }
    uint32_t incl = tot;
#pragma unroll
    for (int k = 1; k < 32; k <<= 1) {
        const uint32_t t = __shfl_up_sync(0xFFFFFFFFu, incl, k);
        if (lane >= (uint32_t)k) incl += t;
    }
    if (lane == 31) s_wsum[warp] = incl;
    __syncthreads();
    if (has_digits) {
        uint32_t first = incl - tot;
        for (uint32_t w = 0; w < warp; ++w) first += s_wsum[w];
#pragma unroll
        for (int k = 0; k < DPT; ++k) {
            const uint32_t d = tid * DPT + k;
            s_dbase[d] = first;
            s_gbase[d] = gstart[k] - first;  // wrapping on purpose
            first += sub[k];
        }
    }
    rs_cp_async_wait<0>();  // my pieces of the values have landed
    __syncthreads();
    // ---- 3. the tile, sorted by digit, in shared memory ------------------------------------------------------------------------
    // values up into registers (their buffer becomes the sorted keys), keys across, values down
    uint32_t val[MODE == RS_KEYS ? 1 : ROUNDS];
    if (MODE != RS_KEYS) {
#pragma unroll
        for (int r = 0; r < ROUNDS; ++r) val[r] = RS_OK(r) ? in_val[wbase + 32 * r] : 0;
        __syncthreads();
    }
#pragma unroll
    for (int r = 0; r < ROUNDS; ++r) {
        if (RS_OK(r)) {
            const uint32_t k = in_key[wbase + 32 * r];
            const uint32_t d = (k >> shift) & (ND - 1);
            const uint32_t p = s_dbase[d] + my_cnt[d] + ((r & 1) ? rank2[r >> 1] >> 16 : rank2[r >> 1] & 0xFFFFu);
            s_key[p] = k;
            if (r & 1) rank2[r >> 1] = (rank2[r >> 1] & 0xFFFFu) | p << 16;  // the slot replaces the rank (TILE <= 65 536)
            else rank2[r >> 1] = (rank2[r >> 1] & 0xFFFF0000u) | p;
        }
    }
    __syncthreads();
    if (MODE != RS_KEYS) {
#pragma unroll
        for (int r = 0; r < ROUNDS; ++r)
            if (RS_OK(r)) s_val[(r & 1) ? rank2[r >> 1] >> 16 : rank2[r >> 1] & 0xFFFFu] = val[r];
        __syncthreads();
    }
    // ---- 4. write out: consecutive threads = consecutive slots = (inside a digit) consecutive global addresses ------------------
#pragma unroll
    for (uint32_t p = tid; p < (FULL ? (uint32_t)TILE : tile_n); p += THREADS) {
        const uint32_t k = s_key[p];
        const uint32_t dst = s_gbase[(k >> shift) & (ND - 1)] + p;
        if (MODE == RS_PAIRS) {
            keys_out[dst] = k;
            vals_out[dst] = s_val[p];
        } else if (MODE == RS_PACK) {
            keys_out[dst] = (k >> (shift + DB)) << aux | s_val[p];
        } else {
            vals_out[dst] = k & aux;
        }
    }
#undef RS_OK
}

template <int DB, int THREADS, int ROUNDS, int MINB, int MODE>
__global__ void __launch_bounds__(THREADS, MINB) radix_scatter_kernel(const uint32_t* __restrict__ keys_in,
                                                                      const uint32_t* __restrict__ vals_in, uint64_t n_cap,
                                                                      const uint64_t* __restrict__ d_n, int shift,
                                                                      uint32_t n_tiles, const uint32_t* __restrict__ bucket_start,
                                                                      uint32_t* __restrict__ keys_out, uint32_t* __restrict__ vals_out,
                                                                      uint32_t aux) {
    constexpr int TILE = THREADS * ROUNDS;
    static_assert((1 << DB) % THREADS == 0 || (1 << DB) < THREADS, "digits must divide over the threads");
    static_assert(ROUNDS % 4 == 0, "ranks are packed in pairs, the tile is staged in 16-byte pieces");
    const uint64_t n = d_n ? min((uint64_t)*d_n, n_cap) : n_cap;
    extern __shared__ __align__(16) uint32_t s_mem[];
    __shared__ uint32_t s_wsum[THREADS / 32];
    const uint64_t tile0 = (uint64_t)blockIdx.x * TILE;
    if (tile0 >= n) return;
    const uint32_t tile_n = (uint32_t)min((uint64_t)TILE, n - tile0);
    if (tile_n == TILE)
        rs_scatter_tile<DB, THREADS, ROUNDS, MODE, true>(keys_in, vals_in, tile0, tile_n, shift, n_tiles, bucket_start, keys_out, vals_out, aux, s_mem, s_wsum);
    else
        rs_scatter_tile<DB, THREADS, ROUNDS, MODE, false>(keys_in, vals_in, tile0, tile_n, shift, n_tiles, bucket_start, keys_out, vals_out, aux, s_mem, s_wsum);
}

static size_t radix_scatter_smem(int width, const RsShape& sh) {
    const size_t nd = (size_t)1 << width, tile = (size_t)sh.threads * sh.rounds;
    return 8 * tile + 8 * nd + 2 * nd * (size_t)(sh.threads / 32);
}

// one pass = histogram (or the caller's own, when it has more to count), scan, scatter
template <int DB, int S, int MODE>
static cudaError_t launch_radix_pass(gtgpu_ctx* ctx, const uint32_t* ki, const uint32_t* vi, uint64_t n, const uint64_t* d_n, int shift,
                                     uint32_t tiles, uint32_t* hist, uint32_t* starts, void* scan_tmp, uint32_t* ko, uint32_t* vo,
                                     uint32_t aux, bool hist_done, int32_t* status) {
    constexpr RsShape sh = RS_SHAPES[S];
    constexpr int TILE = sh.threads * sh.rounds;
    auto kern = radix_scatter_kernel<DB, sh.threads, sh.rounds, sh.min_blocks, MODE>;
    const size_t smem = radix_scatter_smem(DB, sh);
    // > 48 KB of dynamic shared memory is an opt-in per kernel and per device: set it on every call (cheap)
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    if (!hist_done) {
        radix_hist_kernel<DB, TILE><<<tiles, RS_HIST_THREADS, 0, ctx->stream>>>(ki, n, d_n, shift, tiles, hist);
        ctx->launches++;
    }
    *status = exclusive_scan<uint32_t>(ctx, hist, starts, ((uint64_t)1 << DB) * tiles, scan_tmp);
    if (*status != GTGPU_OK) return cudaSuccess;
    kern<<<tiles, sh.threads, smem, ctx->stream>>>(ki, vi, n, d_n, shift, tiles, starts, ko, vo, aux);
    ctx->launches++;
    return cudaGetLastError();
}

template <int S>
static cudaError_t launch_radix_pass_s(int width, gtgpu_ctx* ctx, const uint32_t* ki, const uint32_t* vi, uint64_t n,
                                       const uint64_t* d_n, int shift, uint32_t tiles, uint32_t* hist, uint32_t* starts, void* scan_tmp,
                                       uint32_t* ko, uint32_t* vo, int32_t* status) {
    if (width == 8) return launch_radix_pass<8, S, RS_PAIRS>(ctx, ki, vi, n, d_n, shift, tiles, hist, starts, scan_tmp, ko, vo, 0, false, status);
    return launch_radix_pass<9, S, RS_PAIRS>(ctx, ki, vi, n, d_n, shift, tiles, hist, starts, scan_tmp, ko, vo, 0, false, status);
}

// passes and digit width for `bits` significant key bits: as few passes as 9-bit digits allow, 8-bit digits otherwise
void radix_plan(int bits, int* passes, int* width) {
    *passes = (bits + 8) / 9;
    *width = ((bits + *passes - 1) / *passes) <= 8 ? 8 : 9;
}

static uint64_t rs_min_tile() {
    uint64_t t = ~0ull;
    for (const RsShape& s : RS_SHAPES) t = std::min<uint64_t>(t, (uint64_t)s.threads * s.rounds);
    return t;
}

// sized for the smallest tile any shape uses (the shape is a run-time choice)
size_t radix_sort_temp_bytes(uint64_t n) {
    const uint64_t tiles = (n + rs_min_tile() - 1) / rs_min_tile();
    const uint64_t table = 512 * tiles;
    return (size_t)(table * 4 * 2 + exclusive_scan_temp_bytes(table, 4) + 256);
}

// Sorts by bits [0, bits) of the key; higher bits are ignored (except below bit 8: a single 8-bit pass for bits < 8 sorts by
// bits [0, 8), callers pass keys < 2^bits).  keys/vals ping-pong between the a and b buffers; *result_in_b tells where the
// sorted data ended up.  n < 2^32.
// d_n (optional, device): the real element count when only the device knows it; n is then the capacity the grid is sized for.
int32_t radix_sort_pairs(gtgpu_ctx* ctx, uint64_t n, uint32_t* keys_a, uint32_t* vals_a, uint32_t* keys_b, uint32_t* vals_b,
                         int bits, void* d_temp, int* result_in_b, const uint64_t* d_n) {
    *result_in_b = 0;
    if (n == 0 || bits <= 0) return GTGPU_OK;
    if (n >= 0xFFFFFFFFull) return fail(GTGPU_ERR_UNSUPPORTED, "radix_sort_pairs: too many elements");
    int passes, width;
    radix_plan(std::min(bits, 32), &passes, &width);
    const int shape = rs_shape_index();
    const uint64_t tile = (uint64_t)RS_SHAPES[shape].threads * RS_SHAPES[shape].rounds;
    const uint32_t tiles = (uint32_t)((n + tile - 1) / tile);
    // the table layout of radix_sort_temp_bytes: two tables of 512 words per (smallest) tile, then the scan's own scratch
    const uint64_t cap_tiles = (n + rs_min_tile() - 1) / rs_min_tile();
    uint32_t* hist = reinterpret_cast<uint32_t*>(d_temp);
    uint32_t* starts = hist + 512ull * cap_tiles;
    void* scan_tmp = starts + 512ull * cap_tiles;
    uint32_t *ki = keys_a, *vi = vals_a, *ko = keys_b, *vo = vals_b;
    for (int p = 0, shift = 0; p < passes; ++p, shift += width) {
        // the last digit ends at bit `bits` (overlapping the one before it: the earlier passes already ordered the shared
        // bits, so the stable pass keeps that order), so no key bit at or above `bits` takes part in the order
        if (p == passes - 1 && passes > 1) shift = std::min(bits, 32) - width;
        int32_t status = GTGPU_OK;
        cudaError_t e = cudaErrorInvalidValue;
        switch (shape) {
#define GT_RS_CASE(S)                                                                                                              \
    case S:                                                                                                                        \
        e = launch_radix_pass_s<S>(width, ctx, ki, vi, n, d_n, shift, tiles, hist, starts, scan_tmp, ko, vo, &status);        \
        break;
            GT_RS_CASE(0) GT_RS_CASE(1) GT_RS_CASE(2)
#undef GT_RS_CASE
        }
        static_assert(RS_N_SHAPES == 3, "one case per shape");
        GT_TRY(status);
        GT_CUDA(e);
        std::swap(ki, ko);
        std::swap(vi, vo);
        *result_in_b ^= 1;
    }
    return GTGPU_OK;
}

// ---- stable group-by of values by key: two passes, the second one over packed words ------------------------------------------
// For keys of 10-18 bits whose upper digit fits next to the value in 32 bits (C5: 17-bit barcodes, 20-bit tokens).  Pass 1
// sorts the pairs by the low digit and writes (upper digit << value bits | value); pass 2 sorts those words by the upper digit
// and writes the bare values.  The sorted keys never exist, so the group offsets come from counts: pass 1's output is ordered
// by low digit, G[lo] = where digit lo starts in it; a tile of pass 2 that lies inside one low digit (all but <= 2^w of them)
// knows the full key of every element from its upper digit alone, and its histogram — which pass 2 needs anyway — is added
// to the per-key counts with one atomic per (tile, upper digit); tiles across a boundary look every element's position up.
__global__ void rs_group_prepare_kernel(const uint32_t* __restrict__ starts, uint32_t n_tiles, uint32_t n_lo, uint64_t n_cap,
                                        const uint64_t* __restrict__ d_n, uint32_t tile, uint32_t* __restrict__ G,
                                        uint32_t* __restrict__ tile_lo, uint64_t* __restrict__ d_total) {
    // G[lo] = first position of low digit lo in pass 1's output (= its bucket of tile 0), G[n_lo] = n; every block keeps a copy
    __shared__ uint32_t s_G[513];
    const uint64_t n = d_n ? min((uint64_t)*d_n, n_cap) : n_cap;
    for (uint32_t lo = threadIdx.x; lo <= n_lo; lo += blockDim.x) {
        const uint32_t g = lo < n_lo ? starts[(uint64_t)lo * n_tiles] : (uint32_t)n;
        s_G[lo] = g;
        if (blockIdx.x == 0) G[lo] = g;
    }
    if (blockIdx.x == 0 && threadIdx.x == 0 && d_total) *d_total = (d_n && *d_n > n_cap) ? ~0ull : n;
    __syncthreads();
    // tile_lo[t] = low digit of the tile's first element | 1 << 31 when its last element belongs to another one
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n_tiles) return;
    const uint64_t first = (uint64_t)t * tile, last = min(first + tile, n);
    if (first >= n) {
        tile_lo[t] = 0;
        return;
    }
    uint32_t a = 0, b = n_lo;  // largest lo with G[lo] <= first
    while (b - a > 1) {
        const uint32_t m = (a + b) >> 1;
        if (s_G[m] <= first) a = m;
        else b = m;
    }
    tile_lo[t] = a | (last > s_G[a + 1] ? 0x80000000u : 0u);
}

template <int DB, int TILE>
__global__ void __launch_bounds__(RS_HIST_THREADS) radix_hist_group_kernel(const uint32_t* __restrict__ keys, uint64_t n_cap,
                                                                           const uint64_t* __restrict__ d_n, int shift,
                                                                           uint32_t n_tiles, uint32_t* __restrict__ hist,
                                                                           const uint32_t* __restrict__ tile_lo,
                                                                           const uint32_t* __restrict__ G, uint32_t n_lo, int w,
                                                                           unsigned long long* __restrict__ key_count, uint32_t n_keys) {
    constexpr uint32_t ND = 1u << DB;
    constexpr int WARPS = RS_HIST_THREADS / 32;
    constexpr int ROUNDS = (TILE + RS_HIST_THREADS - 1) / RS_HIST_THREADS;
    const uint64_t n = d_n ? min((uint64_t)*d_n, n_cap) : n_cap;
    __shared__ uint32_t s_hist[WARPS / 2][ND];
    for (uint32_t i = threadIdx.x; i < (WARPS / 2) * ND; i += RS_HIST_THREADS) (&s_hist[0][0])[i] = 0;
    __syncthreads();
    const uint64_t base = (uint64_t)blockIdx.x * TILE;
    const uint64_t lim = min(n, base + TILE);
    const uint32_t tl = tile_lo[blockIdx.x];
    uint32_t* mine = s_hist[(threadIdx.x >> 5) >> 1];
    uint32_t key[ROUNDS];
#pragma unroll
    for (int k = 0; k < ROUNDS; ++k) {
        const uint64_t i = base + (uint64_t)k * RS_HIST_THREADS + threadIdx.x;
        key[k] = i < lim ? __ldcs(keys + i) : 0;
    }
#pragma unroll
    for (int k = 0; k < ROUNDS; ++k) {
        const uint64_t i = base + (uint64_t)k * RS_HIST_THREADS + threadIdx.x;
        if (i < lim) {
            const uint32_t d = (key[k] >> shift) & (ND - 1);
            atomicAdd(&mine[d], 1u);
            if (tl >> 31) {  // a tile across a low-digit boundary: this element's own low digit, from its position
                uint32_t a = tl & 0x7FFFFFFFu, b = n_lo;
                while (b - a > 1) {
                    const uint32_t m = (a + b) >> 1;
                    if (__ldg(G + m) <= i) a = m;
                    else b = m;
                }
                if ((((uint64_t)d << w) | a) < n_keys) atomicAdd(key_count + (((uint64_t)d << w) | a), 1ull);  // (keys >= n_keys: caller's bug, not counted)
            }
        }
    }
    __syncthreads();
    for (uint32_t d = threadIdx.x; d < ND; d += RS_HIST_THREADS) {
        uint32_t t = 0;
#pragma unroll
        for (int k = 0; k < WARPS / 2; ++k) t += s_hist[k][d];
        hist[(uint64_t)d * n_tiles + blockIdx.x] = t;
        if (t && !(tl >> 31) && (((uint64_t)d << w) | tl) < n_keys) atomicAdd(key_count + (((uint64_t)d << w) | tl), (unsigned long long)t);
    }
}

static int rs_bits_for(uint64_t n_values) {
    int b = 1;
    while (b < 63 && (1ull << b) < n_values) ++b;
    return b;
}

bool radix_group_fits(uint32_t n_keys, uint32_t max_val) {
    const char* e = getenv("GTGPU_NO_GROUP_SORT");
    if (e && *e == '1') return false;
    int passes, width;
    const int bits = rs_bits_for(n_keys);
    radix_plan(bits, &passes, &width);
    return passes == 2 && (bits - width) + rs_bits_for((uint64_t)max_val + 1) <= 32;
}

static uint64_t rs_group_tiles(uint64_t n) {
    constexpr uint64_t tile = (uint64_t)RS_SHAPES[0].threads * RS_SHAPES[0].rounds;
    return (n + tile - 1) / tile;
}

// scratch of radix_group_values for n elements and n_keys keys (includes radix_sort_temp_bytes(n))
size_t radix_group_temp_bytes(uint64_t n, uint32_t n_keys) {
    return radix_sort_temp_bytes(n) + (size_t)(520 + rs_group_tiles(n) + 8) * 4 + ((size_t)n_keys + 2) * 8 +
           exclusive_scan_temp_bytes((uint64_t)n_keys + 1, 8) + 64;
}

// vals_out = the values ordered by key (stable), out_offsets[k] = number of elements with a key < k for k in [0, n_keys],
// *d_total (optional) = the element count, ~0 when *d_n exceeded n_cap.  keys < n_keys, vals <= max_val, radix_group_fits.
// packed_tmp: n_cap words; keys / vals are only read.  All on the ctx stream, no host synchronisation.
int32_t radix_group_values(gtgpu_ctx* ctx, uint64_t n_cap, const uint32_t* keys, const uint32_t* vals, uint32_t* packed_tmp,
                           uint32_t* vals_out, uint32_t n_keys, uint32_t max_val, void* d_temp, const uint64_t* d_n,
                           uint64_t* out_offsets, uint64_t* d_total) {
    if (n_cap == 0 || n_cap >= 0xFFFFFFFFull) return fail(GTGPU_ERR_UNSUPPORTED, "radix_group_values: element count");
    if (!radix_group_fits(n_keys, max_val)) return fail(GTGPU_ERR_INVALID, "radix_group_values: keys and values do not pack");
    constexpr int S = 0;  // the default shape; the histogram tile below must be the scatter's
    constexpr int TILE = RS_SHAPES[S].threads * RS_SHAPES[S].rounds;
    int passes, w;
    const int bits = rs_bits_for(n_keys);
    radix_plan(bits, &passes, &w);
    const int hw = bits - w, tb = rs_bits_for((uint64_t)max_val + 1);
    const uint32_t tiles = (uint32_t)rs_group_tiles(n_cap);
    const uint64_t cap_tiles = (n_cap + rs_min_tile() - 1) / rs_min_tile();
    uint32_t* hist = reinterpret_cast<uint32_t*>(d_temp);
    uint32_t* starts = hist + 512ull * cap_tiles;
    void* scan_tmp = starts + 512ull * cap_tiles;
    char* aux = reinterpret_cast<char*>(d_temp) + ((radix_sort_temp_bytes(n_cap) + 15) & ~(size_t)15);
    uint32_t* G = reinterpret_cast<uint32_t*>(aux);
    uint32_t* tile_lo = G + 520;
    unsigned long long* key_count = reinterpret_cast<unsigned long long*>(aux + (((size_t)(520 + tiles) * 4 + 15) & ~(size_t)15));
    void* scan_tmp2 = key_count + n_keys + 2;
    cudaStream_t st = ctx->stream;
    GT_CUDA(cudaMemsetAsync(key_count, 0, ((size_t)n_keys + 1) * 8, st));
    int32_t status = GTGPU_OK;
    // pass 1: pairs by the low digit -> packed words
    cudaError_t e = w == 8 ? launch_radix_pass<8, S, RS_PACK>(ctx, keys, vals, n_cap, d_n, 0, tiles, hist, starts, scan_tmp, packed_tmp, nullptr, (uint32_t)tb, false, &status)
                           : launch_radix_pass<9, S, RS_PACK>(ctx, keys, vals, n_cap, d_n, 0, tiles, hist, starts, scan_tmp, packed_tmp, nullptr, (uint32_t)tb, false, &status);
    GT_TRY(status);
    GT_CUDA(e);
    rs_group_prepare_kernel<<<(tiles + 255) / 256, 256, 0, st>>>(starts, tiles, 1u << w, n_cap, d_n, TILE, G, tile_lo, d_total);
    // pass 2: packed words by the upper digit -> values; its histogram also counts the keys
    const uint32_t mask = tb >= 32 ? 0xFFFFFFFFu : (1u << tb) - 1;
    if (hw <= 8) {
        radix_hist_group_kernel<8, TILE><<<tiles, RS_HIST_THREADS, 0, st>>>(packed_tmp, n_cap, d_n, tb, tiles, hist, tile_lo, G, 1u << w, w, key_count, n_keys);
        e = launch_radix_pass<8, S, RS_KEYS>(ctx, packed_tmp, nullptr, n_cap, d_n, tb, tiles, hist, starts, scan_tmp, nullptr, vals_out, mask, true, &status);
    } else {
        radix_hist_group_kernel<9, TILE><<<tiles, RS_HIST_THREADS, 0, st>>>(packed_tmp, n_cap, d_n, tb, tiles, hist, tile_lo, G, 1u << w, w, key_count, n_keys);
        e = launch_radix_pass<9, S, RS_KEYS>(ctx, packed_tmp, nullptr, n_cap, d_n, tb, tiles, hist, starts, scan_tmp, nullptr, vals_out, mask, true, &status);
    }
    ctx->launches += 2;
    GT_TRY(status);
    GT_CUDA(e);
    GT_TRY(exclusive_scan<unsigned long long>(ctx, key_count, reinterpret_cast<unsigned long long*>(out_offsets), (uint64_t)n_keys + 1, scan_tmp2));
    return GTGPU_OK;
}

}  // namespace gtgpu
