// common.cuh — shared declarations for libgtars_gpu.so (sm_100a).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include <algorithm>
#include <functional>
#include <map>
#include <memory>
#include <mutex>
#include <string>
#include <utility>
#include <vector>

#include "../../../include/gtars_gpu.h"

namespace gtgpu {

// ---- error plumbing ---------------------------------------------------------------------------------------
void set_error(const std::string& msg);
int32_t fail(int32_t code, const std::string& msg);

#define GT_CUDA(expr)                                                                                   \
    do {                                                                                                \
        cudaError_t _e = (expr);                                                                        \
        if (_e != cudaSuccess)                                                                          \
            return ::gtgpu::fail(GTGPU_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(_e));   \
    } while (0)

// Nothing may unwind across the C ABI (the callers are Rust / ctypes): every extern "C" entry point is a function-try-block
// that ends in GT_CATCH — std::bad_alloc becomes GTGPU_ERR_NOMEM, anything else GTGPU_ERR_INVALID, message in last_error.
int32_t translate_exception() noexcept;
#define GT_CATCH catch (...) { return ::gtgpu::translate_exception(); }

#define GT_TRY(expr)                   \
    do {                               \
        int32_t _s = (expr);           \
        if (_s != GTGPU_OK) return _s; \
    } while (0)

// ---- device-side view of an index -----------------------------------------------------------------------------
// One *segment* = one (chromosome, AIList component) run of intervals, start-sorted, with the running max of
// its ends (pmax).  Bits has exactly one segment per chromosome.  All arrays are SoA, 32-bit coordinates.
// Every sorted array that gets searched has a bin LUT in front of it: lut[b] = lower_bound(arr, b << shift),
// so a search is one LUT read (two adjacent words) plus a bisection inside one bin (0–3 probes for peak-like
// universes).  The LUTs and the arrays of a 1 M-region universe are ≈ 25 MB and stay L2-resident.
struct SegMeta {      // 32 bytes, read as two 128-bit loads
    uint32_t off;     // first interval of this segment in starts/ends/pmax/vals
    uint32_t len;
    uint32_t lut_s;   // offset of the LUT over starts (nb_s + 1 entries, segment-local indices)
    uint32_t nb_s;
    uint32_t lut_p;   // offset of the LUT over pmax
    uint32_t nb_p;
    uint32_t mono;    // 1 when ends are non-decreasing in segment order (pmax == ends: every candidate is a hit)
    uint32_t pad;
};

struct ChromMeta {    // 32 bytes
    uint32_t seg_begin, seg_end;  // segments of this chromosome (component order)
    uint32_t off, len;            // chromosome range in cs_starts / cs_ends
    uint32_t lut_cs, nb_cs;       // rank LUT (64-bit entries) over the chromosome's independently sorted starts
    uint32_t lut_ce, nb_ce;       // rank LUT over the chromosome's independently sorted ends
};

// Bin table (the fast path of find/tokenize).  Window b of a chromosome is the two-bin range
// [b << bt_shift, (b+2) << bt_shift); bt_lut[b] names the run of start-sorted intervals that touch it as
// (first << 2) | n.  A query that STARTS in bin b and ends inside that window (any query up to one bin wide) finds
// all its candidates, already in reference order, with one 4-byte LUT load and one or two adjacent 16-byte entry
// loads.  The LUT (4 B/bin) plus the entries (16 B/interval) of a 1 M-region universe are 28 MB and stay resident
// in one die's half of the L2.  Windows with more than two candidates or a non-contiguous candidate run,
// chromosomes with several AIList components or with start > end intervals, wider or degenerate queries all fall
// back to the LUT + walk path below, so results never depend on the table.
// Window word encodings:  0 = empty;  (first << 2) | n, n in {1,2} = direct run;  BT_POOL_FLAG | (offset << 4) | n,
// n in 1..BT_POOL_MAX (15) = candidate list bt_pool[offset .. offset+n) of entry indices, stored in the backend's emission
// order (covers nested intervals and multi-component AIList chromosomes);  BT_OVERFLOW = more candidates than that.
#define BT_OVERFLOW 0xFFFFFFFFu
#define BT_POOL_FLAG 0x80000000u
#define BT_POOL_MAX 15u   // candidates a pool list may hold (4-bit length field)
#define BT_POOL_SHIFT 4   // word = BT_POOL_FLAG | offset << BT_POOL_SHIFT | n
#define BT_SEMI_MAX 7u    // per-query hit count up to which a warp keeps packed offsets (row sums fit a byte)
#define BT_GENERIC_CHROM 0x80000000u  // in ChromBT.n_bins: this chromosome always takes the generic path
#define BT_MULTI_COMP 0x40000000u     // in ChromBT.n_bins: several AIList components (lists of different windows cannot be merged)
#define BT_NBINS_MASK 0x3FFFFFFFu
#define BT_MAX_WINDOWS 8u             // a query may span this many two-bin windows before it goes to the generic walk

// Window records (bt_rec, 16 bytes per bin) are what the fused kernel's fast path reads: the window's one or two
// candidates INLINE, so a query is resolved by ONE 16-byte gather instead of a window word followed by an entry gather
// (measured: 10.9 -> 9.8 ms per 1e9 queries; an 8-byte record that left two-candidate windows to bt_ent was slower).
// Coordinates are relative to the window base (b << bt_shift) and clamped to [0, 2^(bt_shift+1)]: a fast-path query
// starts in bin b and ends inside the window, so the clamped values compare (and overlap-measure) exactly like the
// absolute ones; bt_shift <= 13 keeps them below 2^15.  A candidate is ONE precomputed word:
//   word 0 / 2 = ((e_rel + 0x7FFF) << 16) - s_rel      (absent candidate: e_rel = s_rel = 0, i.e. BT_REC_EMPTY)
//   word 1 / 3 = val of that candidate
// A window query (s_rel = start - base < 2^shift, d = end - 1 - base < 2^(shift+1)) hits the candidate iff
// s_rel_c <= d and s_rel <= e_rel_c - 1, i.e. iff bits 15 and 31 of
//   T = word + ((d + 0x8000) - (s_rel << 16))  =  [ (e_rel_c - 1 + 0x8000) - s_rel ] << 16  |  [ (d + 0x8000) - s_rel_c ]
// are both set (neither half can borrow or carry: every operand is below 2^15) — one add and one logic op per candidate
// (round 2: bit fields that had to be shifted and masked apart cost 7 instructions per candidate; 5.88 -> 5.75 ms).
// The bp filter (min_overlap > 1) recovers the coordinates: s_rel_c = -word mod 2^16, e_rel_c from the upper half.
//   pool list / overflow window: word 0 = BT_REC_SLOW, word 1 = the window's bt_lut word (list offset and length, or
//   BT_OVERFLOW), word 2 = BT_REC_EMPTY.
// bt_lut / bt_ent / bt_pool stay the slow path's view of the same windows (pool lists, multi-window queries).
#define BT_REC_WORDS 4
#define BT_REC_MAX_SHIFT 13u
#define BT_REC_EMPTY 0x7FFF0000u
#define BT_REC_SLOW 0xFFFFFFFFu

struct ChromBT {         // 8 bytes
    uint32_t off;        // first bin record of this chromosome
    uint32_t n_bins;     // bins beyond this hold nothing; BT_GENERIC_CHROM = no table
};

struct IndexView {
    const ChromBT* chrom_bt;
    const uint32_t* bt_lut;
    const uint32_t* bt_rec;
    const uint32_t* bt_pool;
    const uint4* bt_ent;
    uint32_t bt_shift;
    const ChromMeta* chroms;
    const SegMeta* segs;
    const uint32_t* starts;
    const uint32_t* ends;
    const uint32_t* pmax;
    const uint32_t* vals;
    const uint32_t* cs_starts;
    const uint32_t* cs_ends;
    const uint32_t* lut;
    // Rank LUT for the counting identity: one 64-bit word per bin = base index (32) | count (3; 7 = more than fit) |
    // the in-bin offsets of up to rank_inline entries (rank_shift bits each).  lower_bound(key) is ONE 8-byte load:
    // base + #{inline offsets < key's in-bin offset}.  With about one bin per interval a 50 M-interval database costs
    // one DRAM sector per search instead of a LUT read plus a bisection over 32-byte sectors of the sorted array.
    const unsigned long long* rank_lut;
    uint32_t rank_shift, rank_inline;
    // The rank LUT holds the starts LUTs of all chromosomes back to back, then (from word rank_ends_off) their ends LUTs.
    // rank_lin[c] = {first starts word << rank_shift, starts bins << rank_shift, first ends word (inside the ends block) <<
    // rank_shift, ends bins << rank_shift}: lin = .x + min(key, .y) names the LUT word (lin >> rank_shift) AND the in-bin
    // offset (low bits) of a starts search without the chromosome — 4 bytes per search for the bucketed counting pass.
    // nullptr when a block's linearised span does not fit 32 bits (that pass is then not used).
    const uint4* rank_lin;
    uint32_t rank_ends_off;
    uint32_t n_chroms;
    uint32_t shift;
    uint32_t descending;  // 1 = AIList emission order (descending position inside a segment)
    uint32_t proper;      // 1 = every interval has start <= end (Bits identity usable)
};

// ---- host-side objects ---------------------------------------------------------------------------------------
struct DevBuffer {
    void* ptr = nullptr;
    size_t cap = 0;
};

struct PinnedBlock {
    void* ptr = nullptr;
    size_t cap = 0;
};

}  // namespace gtgpu

struct gtgpu_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    cudaStream_t copy_in = nullptr, copy_out = nullptr;
    uint64_t launches = 0;
    int sm_count = 148;
    std::mutex mu;
    std::vector<gtgpu::DevBuffer> scratch;       // grow-only device scratch, indexed by role
    std::mutex pinned_mu;                         // guards pinned_free; a leaf lock: nothing else is locked while it is held
    std::vector<gtgpu::PinnedBlock> pinned_free;  // cache of pinned result blocks
    uint64_t* h_scalars = nullptr;                // small pinned mailbox
    void* comm = nullptr;                         // gtgpu::Comm (NCCL), set by gtgpu_comm_init
    // Multi-device group (gtgpu_init_multi): peers[0] == this, one ctx per device; empty for a plain single-device ctx.
    // Group-wide calls (index build, batch queries, IGD counts) shard their work over the peers; a peer that is not
    // peers[0] is owned by the group and shut down with it.
    std::vector<gtgpu_ctx*> peers;
    std::mutex group_mu;                          // serialises group-wide calls
    bool group_comm_tried = false;                // in-process NCCL communicators (ncclCommInitAll) were set up / attempted
    int fused_bps[2][12] = {{0}, {0}};  // resident CTAs per SM of the fused find variants
    const void* l2_window_owner = nullptr;        // the index whose window table the stream's access-policy window covers
    bool timing = false;                          // bracket dominant kernels with events
    std::vector<cudaEvent_t> ev_begin, ev_end;
    uint32_t ev_used = 0;
    void time_begin();
    void time_end();
    int32_t scratch_get(int role, size_t bytes, void** out);
    int32_t pinned_get(size_t bytes, gtgpu::PinnedBlock* out);  // both take pinned_mu: callable with or without mu held
    void pinned_put(gtgpu::PinnedBlock b);
};

namespace gtgpu {
// grid of a grid-stride kernel of 256-thread blocks over n items: one block per 256 items, at most 16 per SM
inline int grid_for(const gtgpu_ctx* ctx, uint64_t n) {
    return (int)std::max<uint64_t>(1, std::min<uint64_t>((n + 255) / 256, (uint64_t)ctx->sm_count * 16));
}
}  // namespace gtgpu

struct gtgpu_buf {
    gtgpu_ctx* ctx = nullptr;
    gtgpu::PinnedBlock block;
    uint64_t len = 0;  // elements
    uint32_t elem_size = 4;
};

namespace gtgpu {
// A result buffer the library still owns: dropping it returns the block to its ctx's cache (gtgpu_buf_free).  Hand it to the
// caller with release() once the call can no longer fail.  A buffer with a D2H copy in flight must not be dropped before the
// stream that carries the copy is synchronised.
struct BufFree {
    void operator()(gtgpu_buf* b) const { gtgpu_buf_free(b); }
};
using BufPtr = std::unique_ptr<gtgpu_buf, BufFree>;
// len elements of elem_size bytes; fails with a status, never with an exception (a caller may hold a buffer with a copy in flight)
int32_t buf_new(gtgpu_ctx* ctx, uint64_t len, uint32_t elem_size, BufPtr* out);
// buf_new, then the D2H copy of the buffer from d_src enqueued on st, not synchronised.  A copy that cannot be enqueued fails
// with GTGPU_ERR_CUDA and the CUDA error text alone in last_error, for the caller to put its own name in front of.
int32_t buf_from_device(gtgpu_ctx* ctx, const void* d_src, uint64_t len, uint32_t elem_size, cudaStream_t st, BufPtr* out);
}  // namespace gtgpu

struct gtgpu_index {
    gtgpu_ctx* ctx = nullptr;
    int32_t kind = 0;
    gtgpu::IndexView view{};
    std::vector<void*> allocs;
    uint64_t n_intervals = 0, n_segments = 0, device_bytes = 0, max_components = 0;
    uint64_t bt_bins = 0, bt_overflow_bins = 0, bt_pool_windows = 0;
    uint64_t rank_lut_len = 0;  // 64-bit words in view.rank_lut (bucket boundaries of the partitioned count)
    uint32_t max_val = 0;  // largest val of any interval (bounds the radix passes of the scoring group-by)
    bool bt_clean = false;            // every window is a plain record: the lean find kernel can serve the index
    bool lean_off = false;            // the lean kernel had to fall back on this index before
    uint32_t* h_lean_probe = nullptr; // pinned copy of the last launch's lean flag (read lazily, never waited for)
    // Group index (built on a multi-device ctx): replicas[r] lives on ctx->peers[r]; replicas[0] == this.
    std::vector<gtgpu_index*> replicas;
};

// gtars-igd database on the device (igd.cu).  A group igd (built on a multi-device ctx) is a header without device data:
// shards[r] holds the region sets [r * C, min((r + 1) * C, n_files)) on ctx->peers[r], C = ceil(n_files / devices).
struct gtgpu_igd {
    gtgpu_ctx* ctx = nullptr;
    uint64_t n_files = 0, n_records = 0;
    uint32_t n_chroms = 0, shift = 0;
    // per chromosome (n_chroms + 1 offsets into the record arrays; LUT offsets / bin counts)
    std::vector<uint32_t> h_off;
    uint32_t *d_off = nullptr, *d_lut_s_off = nullptr, *d_nb_s = nullptr, *d_lut_p_off = nullptr, *d_nb_p = nullptr;
    int32_t *d_start = nullptr, *d_end = nullptr, *d_pmax = nullptr, *d_psame1 = nullptr;
    uint32_t *d_file = nullptr, *d_lut = nullptr;
    std::map<int32_t, int32_t*> psame_by_m;  // psame for every min_overlap asked for so far (derived on the device)
    std::vector<void*> allocs;
    uint64_t device_bytes = 0;
    std::vector<gtgpu_igd*> shards;
    // What gtgpu_igd_serialize needs beyond the records.  Per file: the input's region lines with start < end (as u32) and the
    // wrapping sum of their int32 widths (the .tsv).  Per chromosome: its largest kept end (the contig's tile count), and
    // h_first: the smallest input index of a kept record on it or, when contig_by_file, the smallest file with one (the rank
    // of the contig in the reference's creation order; UINT32_MAX: none).  A shard's values count from its own first file /
    // record (file0 / rec0 in the group's input).
    std::vector<uint64_t> h_file_regions, h_file_widths;
    std::vector<uint32_t> h_first, h_max_end;
    bool contig_by_file = false;
    uint64_t file0 = 0, rec0 = 0;
};

namespace gtgpu {

enum ScratchRole {
    SC_CHR = 0, SC_START, SC_END, SC_BARCODE, SC_OUT_IDS, SC_OUT_IDS2, SC_OUT_OFFS, SC_FILE_OFFS, SC_FILE_TOK,
    SC_FILE_TOK2, SC_TILE_STATUS, SC_TILE_FILE, SC_MISC, SC_COUNTS, SC_IN2_CHR, SC_IN2_START, SC_IN2_END,
    SC_IN3_CHR, SC_IN3_START, SC_IN3_END, SC_SET_ID, SC_MATRIX, SC_ING_0, SC_ING_1, SC_ING_2, SC_ING_3, SC_ING_4, SC_ING_5,
    SC_ING_6, SC_ING_7, SC_GZ_IN, SC_GZ_OUT, SC_GZ_MOFF, SC_GZ_OOFF, SC_GZ_STATUS, SC_CNT_KEYS, SC_CNT_RES, SC_CNT_POS, SC_CNT_RUNS,
    SC_WIN_A, SC_WIN_B, SC_N_ROLES
};

// kernels.cu
#ifndef GT_FUSED_ROWS
#define GT_FUSED_ROWS 4
#endif
#ifndef GT_FUSED_MINBLOCKS
#define GT_FUSED_MINBLOCKS 4
#endif
#ifndef GT_FUSED_BLOCK
#define GT_FUSED_BLOCK 256
#endif
constexpr int FUSED_BLOCK = GT_FUSED_BLOCK;  // threads (8 warps) per tile
constexpr int FUSED_ROWS = GT_FUSED_ROWS;    // queries per thread per tile (striped inside each warp)
constexpr int FUSED_TILE = FUSED_BLOCK * FUSED_ROWS;
constexpr int CHROM_CACHE = 256;             // per-chromosome table entries staged in shared memory

enum CountMode { COUNT_U32 = 0, COUNT_ANY_U8 = 1, COUNT_BITS_RAW_U64 = 2 };

void release_l2_window(gtgpu_ctx* ctx);
int32_t launch_count(gtgpu_index* ix, uint64_t n, const uint32_t* d_chr, const uint32_t* d_start,
                     const uint32_t* d_end, int32_t min_overlap, int mode, void* d_out);

// Workspace the fused kernel needs (device): tile status words + per-tile first-file marks + 2 scalars.
size_t fused_workspace_bytes(uint64_t n);
// d_base (device u64, may be null = 0) is the id offset this launch starts at; *d_total_out receives
// base + ids produced.  d_errflag (device u32) is set to 1 when a tile overflows 32-bit local offsets.
int32_t launch_fused_find(gtgpu_index* ix, uint64_t n, uint64_t n_files, const uint64_t* d_file_offsets,
                          const uint32_t* d_chr, const uint32_t* d_start, const uint32_t* d_end,
                          int32_t min_overlap, uint32_t* d_out_ids, uint64_t ids_capacity,
                          uint64_t* d_out_offsets, uint64_t* d_out_file_tok, void* d_workspace,
                          const uint64_t* d_base, uint64_t* d_total_out, uint32_t* d_errflag, int unk_per_query = 0,
                          uint32_t unk_id = 0, const uint32_t* d_tag_in = nullptr, uint32_t* d_out_tags = nullptr,
                          const uint32_t** tags_pending_if = nullptr);
// d_out_tags (with unk_per_query): out_tags[j] = d_tag_in[query of id j], written by the find itself when the lean kernel
// serves the launch.  *tags_pending_if then points at a device flag that is non-zero iff the launch fell back to the full
// kernel (which writes per-query offsets instead: tag from those); nullptr = the tags were not written at all.
// Per-call [unk] rule: expands raw per-file id runs into d_out, inserting unk_id for files with no ids.
int32_t launch_unk_offsets(gtgpu_ctx* ctx, uint64_t n_files, const uint64_t* d_raw_file_tok,
                           uint64_t* d_out_file_tok, uint64_t* d_n_empty);
int32_t launch_expand_runs(gtgpu_ctx* ctx, uint64_t n_runs, const uint64_t* d_run_offsets, const uint32_t* d_run_chr, uint64_t q0,
                           uint64_t cn, uint32_t* d_out);
int32_t launch_expand_widths(gtgpu_ctx* ctx, uint64_t n, const uint32_t* d_start, const uint16_t* d_w16, uint32_t* d_end,
                             uint64_t n_wide, const uint64_t* d_wide_index, const uint32_t* d_wide_end, uint64_t q0);
int32_t launch_expand_packed(gtgpu_ctx* ctx, uint64_t n, const uint32_t* d_packed, const uint32_t* d_anchors, uint32_t width_bits,
                             uint32_t* d_start, uint32_t* d_end, uint64_t n_exc, const uint64_t* d_exc_index,
                             const uint32_t* d_exc_start, const uint32_t* d_exc_end, uint64_t q0);
int32_t launch_fill_set_ids(gtgpu_ctx* ctx, uint64_t n_sets, const uint64_t* d_set_offsets, uint32_t* d_set_of);
int32_t launch_unk_expand(gtgpu_ctx* ctx, uint64_t n_files, const uint64_t* d_raw_file_tok,
                          const uint64_t* d_out_file_tok, const uint32_t* d_raw_ids, uint32_t unk_id,
                          uint32_t* d_out_ids);

// scoring.cu: fused find over device-resident queries with the optimistic-capacity + exact re-run protocol; the raw
// ids land in scratch SC_OUT_IDS (*d_ids), *total_out is their number.  d_offsets / d_file_tok may be null.
int32_t fused_find_all(gtgpu_index* ix, uint64_t nq, uint64_t n_files, const uint64_t* d_qfo, const uint32_t* d_qc,
                       const uint32_t* d_qs, const uint32_t* d_qe, uint64_t* d_offsets, uint64_t* d_file_tok,
                       uint32_t** d_ids, uint64_t* total_out, int32_t min_overlap = 0);
// scoring.cu: `total` device (key, value) pairs -> CSR, by two stable radix sorts (values of val_bits bits, then keys < n_keys)
// and a run-length encode.  out_key_offsets (host, n_keys + 1) index, per key, its distinct values in ascending order
// (*out_values) and how often each occurs (*out_counts).  d_keys / d_vals are sorted in place and must lie outside the scratch
// this takes (SC_IN2_START, SC_IN2_END, SC_IN3_*, SC_COUNTS, SC_OUT_IDS2, SC_FILE_TOK): a slot that grows is freed.  who names
// the caller in errors.  Synchronises the ctx stream; the caller holds ctx->mu.
int32_t reduce_pairs_csr_locked(gtgpu_ctx* ctx, uint64_t total, uint32_t* d_keys, uint32_t* d_vals, int val_bits, uint32_t n_keys,
                                uint64_t* out_key_offsets, gtgpu_buf** out_values, gtgpu_buf** out_counts, const std::string& who);

// fragments.cu: tokenize_fragment_file over device-resident fragments with dense barcode ids (caller holds ctx->mu)
int32_t tokenize_fragments_core(gtgpu_index* ix, uint64_t n, const uint32_t* d_chr, const uint32_t* d_start, const uint32_t* d_end,
                                uint32_t* d_bc, uint32_t n_barcodes, uint32_t unk_id, uint64_t* out_barcode_offsets, BufPtr* out_ids);
// fragments.cu: count_fragments_by_barcode over the same input: out_barcode_offsets (host, n_barcodes + 1) index each barcode's
// distinct token ids in ascending order (*out_tokens) and their counts (*out_counts); a fragment without a hit counts as unk_id
int32_t count_fragments_core(gtgpu_index* ix, uint64_t n, const uint32_t* d_chr, const uint32_t* d_start, const uint32_t* d_end,
                             const uint32_t* d_bc, uint32_t n_barcodes, uint32_t unk_id, uint64_t* out_barcode_offsets,
                             gtgpu_buf** out_tokens, gtgpu_buf** out_counts);

// sort.cu — hand-written scan / radix sort
size_t exclusive_scan_temp_bytes(uint64_t n, size_t elem);
template <typename T>
int32_t exclusive_scan(gtgpu_ctx* ctx, const T* d_in, T* d_out, uint64_t n, void* d_temp);
int32_t inclusive_max_scan_u64(gtgpu_ctx* ctx, const unsigned long long* d_in, unsigned long long* d_out, uint64_t n, void* d_temp);
size_t radix_sort_temp_bytes(uint64_t n);
int32_t radix_sort_pairs(gtgpu_ctx* ctx, uint64_t n, uint32_t* keys_a, uint32_t* vals_a, uint32_t* keys_b, uint32_t* vals_b,
                         int bits, void* d_temp, int* result_in_b, const uint64_t* d_n = nullptr);
void radix_plan(int bits, int* passes, int* width);
// stable group-by of values by key in two passes, the second over packed words (sort.cu)
bool radix_group_fits(uint32_t n_keys, uint32_t max_val);
size_t radix_group_temp_bytes(uint64_t n, uint32_t n_keys);
int32_t radix_group_values(gtgpu_ctx* ctx, uint64_t n_cap, const uint32_t* keys, const uint32_t* vals, uint32_t* packed_tmp,
                           uint32_t* vals_out, uint32_t n_keys, uint32_t max_val, void* d_temp, const uint64_t* d_n,
                           uint64_t* out_offsets, uint64_t* d_total);

// ingest.cu / inflate.cu (the caller holds ctx->mu)
// 64-bit FNV-1a of n bytes
__host__ __device__ __forceinline__ unsigned long long fnv1a64(const char* p, uint32_t n) {
    unsigned long long h = 1469598103934665603ull;
    for (uint32_t i = 0; i < n; ++i) h = (h ^ (unsigned char)p[i]) * 1099511628211ull;
    return h;
}
struct NameTable {
    const char* blob;             // names back to back
    const uint32_t* offsets;      // n_names + 1
    const unsigned long long* hash;  // FNV-1a of every name, sorted ascending
    const uint32_t* hash_id;      // name id of the k-th sorted hash
    uint32_t n_names;
    const uint32_t* rank;         // lexicographic rank of every name (only when asked for)
    // id of the name s[0, len) with FNV-1a hash h, or GTGPU_UNKNOWN_CHROM
    __device__ uint32_t lookup(unsigned long long h, const char* __restrict__ s, uint32_t len) const {
        uint32_t lo = 0, hi = n_names;
        while (lo < hi) {
            const uint32_t mid = (lo + hi) >> 1;
            if (hash[mid] < h) lo = mid + 1;
            else hi = mid;
        }
        for (; lo < n_names && hash[lo] == h; ++lo) {  // equal hashes: compare the bytes
            const uint32_t id = hash_id[lo], na = offsets[id], nb = offsets[id + 1];
            bool same = nb - na == len;
            for (uint32_t i = 0; same && i < len; ++i) same = blob[na + i] == s[i];
            if (same) return id;
        }
        return GTGPU_UNKNOWN_CHROM;
    }
};
// the caller's chromosome names -> scratch SC_SET_ID; with_rank adds the names' lexicographic ranks (NameTable::rank)
int32_t upload_name_table(gtgpu_ctx* ctx, uint32_t n_names, const char* names, const uint32_t* name_offsets, NameTable* out,
                          bool with_rank = false);
// What the BED line kernel needs to parse a text of several files back to back (ingest_parse_lines_kernel<true>).
struct BedFilesView {
    const unsigned long long* file_offsets = nullptr;  // n_files + 1 byte offsets of the files in the whole text
    uint64_t n_files = 0;
    uint64_t byte0 = 0, line0 = 0;                     // the window's first byte and first line in the whole text
    unsigned long long* first_line = nullptr;          // [f] = text-wide index of file f's first line
    const uint32_t* fstart = nullptr;                  // the window's n_fstart file starts in (0, n_bytes), sorted
    uint32_t n_fstart = 0;
};
// The line formats of the device text parsers; each has its own line kernel, the front end around it is shared.
// BED_LINES: gtgpu_parse_bed's rules, names looked up in the name table.  BED_FILE_LINES: the same per file of a BedFilesView,
// chr = the line's file index, and the chromosome name carried as a key.  Fragments: tokenize_fragment_file needs fields 1
// and 2 as u32 and the barcode (the key); Fragment::from_str (scoring) needs field 4 as well, and the count matrix has no use
// for the barcode.
enum LineFormat { BED_LINES, BED_FILE_LINES, FRAG_TOKENIZE, FRAG_SCORE_MATRIX, FRAG_SCORE_BARCODES };
struct ParsedLines {
    uint32_t n_lines = 0;
    uint32_t bad_line = 0xFFFFFFFFu;  // 0-based index of the first malformed line of the text, or none
    uint32_t n = 0;                   // kept lines (0 when a line was malformed)
    uint32_t *chr = nullptr, *start = nullptr, *end = nullptr;  // scratch SC_CHR / SC_START / SC_END
    unsigned long long* h = nullptr;  // per kept line the key's FNV-1a hash (never 0), byte offset and length in the text
    uint32_t *bo = nullptr, *bl = nullptr;  // (BED_FILE_LINES, FRAG_TOKENIZE, FRAG_SCORE_BARCODES only)
    const uint32_t* breaks = nullptr;       // the line break positions (scratch SC_IN3_END): line i > 0 starts at breaks[i - 1] + 1
    uint32_t* free[5] = {};  // line-sized scratch the caller may reuse (SC_ING_0, SC_ING_1, SC_IN2_CHR, SC_IN2_START, SC_IN2_END)
    void* tmp = nullptr;     // scan temp for line-sized arrays (scratch SC_IN3_START)
    uint32_t* flags = nullptr;  // device words [1..3], zeroed for the caller (scratch SC_MISC)
};
// The line front end: line breaks, the format's one-thread-per-line kernel, compaction of the kept lines.  d_text: 0 < n_bytes
// < 0xFFFFFFF0 bytes of device text, 16-byte aligned; files only for BED_FILE_LINES.  Synchronises the ctx stream.
int32_t parse_lines_locked(gtgpu_ctx* ctx, const char* d_text, uint64_t n_bytes, LineFormat fmt, const NameTable& nt,
                           const BedFilesView& files, ParsedLines* out);
// A device buffer owned by one call, grown while keeping its first `keep` bytes.
struct DevMem {
    void* ptr = nullptr;
    size_t cap = 0;
    DevMem() = default;
    DevMem(const DevMem&) = delete;
    DevMem& operator=(const DevMem&) = delete;
    ~DevMem();
    int32_t reserve(size_t bytes, size_t keep, cudaStream_t st);
    void swap(DevMem& o) { std::swap(ptr, o.ptr); std::swap(cap, o.cap); }
    uint32_t* u32() const { return static_cast<uint32_t*>(ptr); }
};
// The keys of one text over all its windows (barcodes of a fragment file, chromosome names of BED files): dense ids in
// first-appearance order among the kept keys.  keep_all keeps every key; otherwise only those seen on a line whose chr is in
// the name table are kept.  At most max_keys distinct keys are allowed.  record_spans keeps each key's first byte offset in
// the text for finish()'s spans.  who / array_entry name the caller and its array entry point in error messages; key / keys
// name one key and the keys in them.  chr / start / end hold the parsed columns of every kept line, id the key's
// first-appearance index per line, and after finish() the key's dense id (0 for a line of a dropped key).
struct KeyTable {
    const bool keep_all, record_spans;
    const uint64_t max_keys;
    const std::string who, array_entry, key, keys;
    DevMem chr, start, end, id;                                // per line
    DevMem hash, first, soff, klen, known, first_byte, arena;  // per slot (hash 0 = empty), and the keys' bytes
    uint64_t n = 0, distinct = 0, cap = 0, used = 0;
    KeyTable(bool keep_all_, bool record_spans_, uint64_t max_keys_, std::string who_, std::string array_entry_, std::string key_,
             std::string keys_)
        : keep_all(keep_all_), record_spans(record_spans_), max_keys(max_keys_), who(std::move(who_)),
          array_entry(std::move(array_entry_)), key(std::move(key_)), keys(std::move(keys_)) {}
    // byte0: the window's offset in the text; pl carries keys (h / bo / bl)
    int32_t add_window(gtgpu_ctx* ctx, const char* d_text, uint64_t byte0, const ParsedLines& pl, uint32_t n_names);
    // With out_spans (needs record_spans): n_kept (first byte, length) u32 pairs, and out_names / out_name_offsets are untouched.
    // Otherwise *out_names: the kept keys' bytes back to back (elem_size 1); *out_name_offsets: n_kept + 1 u64 offsets into them.
    int32_t finish(gtgpu_ctx* ctx, uint32_t* n_kept, BufPtr* out_names, BufPtr* out_name_offsets, BufPtr* out_spans = nullptr);
};
// ---- the text input of the device parsers -------------------------------------------------------------------------------------
// What an entry point was given: plain text (text, n_bytes), or gzip members (member k = gz[member_offsets[k], member_offsets[k + 1]),
// as gtgpu_gunzip takes them), and for the entry points that take several files, where each file starts: file f =
// text[file_offsets[f], file_offsets[f + 1]) or the members [file_members[f], file_members[f + 1]).  check() holds every argument
// rule of these entry points (GTGPU_ERR_INVALID, "who: ..."); open_text_locked turns a checked input into a Text.
struct TextIn {
    const char* text = nullptr;
    uint64_t n_bytes = 0;
    const uint8_t* gz = nullptr;
    uint64_t n_members = 0;
    const uint64_t* member_offsets = nullptr;
    bool is_gz = false, files = false;
    uint64_t n_files = 0;
    const uint64_t* file_offsets = nullptr;  // plain text of files: n_files + 1 byte offsets
    const uint64_t* file_members = nullptr;  // gzip members of files: n_files + 1 member indices
    static TextIn plain(const char* text, uint64_t n_bytes);
    static TextIn plain(const char* text, uint64_t n_files, const uint64_t* file_offsets);
    static TextIn gzip(uint64_t n_members, const uint8_t* gz, const uint64_t* member_offsets);
    static TextIn gzip(uint64_t n_members, const uint8_t* gz, const uint64_t* member_offsets, uint64_t n_files, const uint64_t* file_members);
    int32_t check(const std::string& who) const;
};
// The text a parser reads: n_bytes at `bytes`, in the caller's host memory (staged to the device by the parser) or, when on_device,
// in device memory (inflated gzip members, read in place).  file_offsets: the files' n_files + 1 byte offsets in the text.
struct Text {
    const char* bytes = nullptr;
    bool on_device = false;
    uint64_t n_bytes = 0;
    uint64_t n_files = 0;
    std::vector<uint64_t> file_offsets;
};
// A checked TextIn as a Text: gzip members are inflated whole into device memory (scratch SC_GZ_OUT, by gunzip_locked) and the
// files' member ranges become byte ranges of that text.  The caller holds ctx->mu.
int32_t open_text_locked(gtgpu_ctx* ctx, const TextIn& in, const std::string& who, Text* out);
// inflate.cu: H2D of gzip members + inflate; the text stays in scratch SC_GZ_OUT
int32_t gunzip_locked(gtgpu_ctx* ctx, uint64_t n_members, const uint8_t* gz, const uint64_t* member_offsets,
                      uint64_t* out_member_offsets, uint8_t** d_text, uint64_t* n_text);

// A fragment text of any size in windows that end right after a '\n' (about GTGPU_INGEST_WINDOW bytes, default 2 GiB).  fn gets
// each window's device bytes, its size, its byte offset in the file and the file-wide index of its first line, and returns
// the window's line count.  Host text is staged through pinned memory, device text read in place.
using WindowFn = std::function<int32_t(const char* d_window, uint64_t n_bytes, uint64_t byte0, uint64_t first_line, uint32_t* n_lines)>;
int32_t for_each_window(gtgpu_ctx* ctx, const Text& t, const std::string& who, const WindowFn& fn);

// The region lines of t.n_files BED files back to back (any total size), parsed on the device in windows: line rules of
// gtgpu_parse_bed per file, chromosome names discovered in first-appearance order.
// On success chr / start / end / file hold the n records in file order (chr = dense name id), file_offsets the files' record
// offsets (n_files + 1), names / name_offsets the n_names chromosome names in id order.  The caller holds ctx->mu.
struct BedFilesRecords {
    DevMem chr, start, end, file;
    uint64_t n = 0;
    std::vector<uint64_t> file_offsets;
    uint32_t n_names = 0;
    BufPtr names, name_offsets;
};
int32_t parse_bed_files_locked(gtgpu_ctx* ctx, const Text& t, const std::string& who, BedFilesRecords* out);
// parse_bed_files_locked for query files: every record's chr in the ids of the caller's names (GTGPU_UNKNOWN_CHROM for a name
// not among them).  *nt: the caller's name table in scratch SC_SET_ID (with_rank adds the names' ranks), uploaded when r->n > 0.
int32_t parse_bed_queries_locked(gtgpu_ctx* ctx, const Text& t, uint32_t n_names, const char* names, const uint32_t* name_offsets,
                                 bool with_rank, const std::string& who, BedFilesRecords* r, NameTable* nt);

// groups (api.cu, comm.cu, igd.cu)
int32_t for_each_device(size_t n_devices, const std::function<int32_t(size_t)>& fn);
void block_range(uint64_t n, uint64_t world, uint64_t r, uint64_t* lo, uint64_t* hi);
int32_t group_comm_ensure(gtgpu_ctx* g);
int32_t igd_count_sharded_impl(gtgpu_ctx* ctx, gtgpu_igd* igd, int32_t binary, uint64_t n_files_global, uint64_t n_sets,
                               const uint64_t* set_offsets, const uint32_t* chr, const uint32_t* start, const uint32_t* end,
                               int32_t min_overlap, uint64_t* out, const std::function<bool(bool)>* before_collective);
// the caller holds igd->ctx->mu
int32_t igd_count_dev_locked(gtgpu_igd* g, bool binary, uint64_t n, const uint32_t* d_set_of, const uint32_t* d_chr,
                             const uint32_t* d_start, const uint32_t* d_end, int32_t m, uint64_t* d_out);

// build.cu — device-side primitives of the index builders
struct LutDesc {       // one bin LUT over arr[arr_off .. arr_off + len): nb + 1 entries written at lut[lut_off ..]
    uint32_t arr_off, len, lut_off, nb;
};
int bits_for_value(uint64_t max_value);
int32_t launch_gather_u32(gtgpu_ctx* ctx, uint64_t n, const uint32_t* d_src, const uint32_t* d_perm, uint32_t* d_out);
int32_t launch_key_offsets(gtgpu_ctx* ctx, uint64_t n, const uint32_t* d_sorted, uint32_t n_keys, uint32_t* d_out);
int32_t launch_build_luts(gtgpu_ctx* ctx, uint32_t n_desc, const LutDesc* d_desc, const uint64_t* d_bin_prefix, uint64_t total_bins,
                          const uint32_t* d_arr, uint32_t shift, uint32_t* d_lut);
// Stable LSD radix sort of a permutation of [0, n) by successive key arrays (least significant key first).
struct PermSorter {
    gtgpu_ctx* ctx = nullptr;
    uint64_t n = 0;
    uint32_t *perm = nullptr, *perm_alt = nullptr;  // perm: the current order
    uint32_t *key = nullptr, *key_alt = nullptr;    // key: the last pass's keys, in the current order
    void* tmp = nullptr;
    uint32_t* d_max = nullptr;
    int32_t init(gtgpu_ctx* ctx, uint64_t n);
    int32_t pass(const uint32_t* d_src, int bits);
    ~PermSorter();
};

}  // namespace gtgpu
