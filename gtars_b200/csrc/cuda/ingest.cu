// ingest.cu — BED text -> sorted SoA queries on the device (SURVEY §8f f4).
//
// Once the find kernel runs at > 1e11 queries/s, parsing "chr\tstart\tend\n" on a host core (~1e8 lines/s) is the
// end-to-end bottleneck by three orders of magnitude.  This file restates RegionSet::try_from
// (gtars-core/src/models/region_set.rs:60-185: line rules, u32 parsing, header / comment rows) and RegionSet::sort
// (:502-505: stable, by chromosome string then start) as kernels over the raw bytes of one (already decompressed) file:
//   1. newline positions: per-64-byte-chunk counts -> hand-written exclusive scan -> positions
//   2. one thread per line: comment / header rules, chromosome name -> dense id (hash + byte compare against the
//      caller's name table), str::parse::<u32>() for start and end; the first malformed line is reported
//   3. compaction of the kept lines (scan + scatter)
//   4. order check; when the file is not already sorted: two stable passes of the hand-written radix sort
//      (start, then chromosome rank) and a gather
// gtgpu_tokenize_bed chains the fused find kernel behind it, so a BED file goes from text to token ids without its
// regions ever existing on the host.  Chromosome names that are not in the table map to GTGPU_UNKNOWN_CHROM and sort
// after every known name (the reference sorts them by their own strings; they produce no output either way).
#include <algorithm>
#include <cstdlib>
#include <cstring>
#include <numeric>
#include <string>
#include <string_view>
#include <thread>
#include <vector>

#include "common.cuh"

namespace gtgpu {

constexpr int INGEST_CHUNK = 64;  // bytes per thread in the newline passes

// first index of the sorted array a[0, n) whose value is >= key
__device__ __forceinline__ uint32_t lower_bound_u32(const uint32_t* __restrict__ a, uint32_t n, uint32_t key) {
    uint32_t lo = 0, hi = n;
    while (lo < hi) {
        const uint32_t mid = (lo + hi) >> 1;
        if (a[mid] < key) lo = mid + 1;
        else hi = mid;
    }
    return lo;
}

// Line breaks: every '\n', and (for a text of several files) the byte in front of a file start p that no '\n' precedes, so that a
// file's last line ends with the file.  fstart: n_fstart sorted window-relative file starts in (0, n_bytes), or none.
__global__ void ingest_count_newlines_kernel(uint64_t n_bytes, const char* __restrict__ text, uint32_t* __restrict__ counts,
                                             const uint32_t* __restrict__ fstart, uint32_t n_fstart) {
    const uint64_t n_chunks = (n_bytes + INGEST_CHUNK - 1) / INGEST_CHUNK;
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t c = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; c < n_chunks; c += stride) {
        const uint64_t a = c * INGEST_CHUNK, b = min(a + INGEST_CHUNK, n_bytes);
        uint32_t k = 0;
        if (b - a == INGEST_CHUNK) {
            const uint4* p = reinterpret_cast<const uint4*>(text + a);  // text is 256-byte aligned device scratch
#pragma unroll
            for (int i = 0; i < INGEST_CHUNK / 16; ++i) {
                const uint4 v = __ldg(p + i);
                const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const uint32_t x = w[j] ^ 0x0A0A0A0Au;  // a zero byte where the text has '\n'
                    k += __popc(~((((x & 0x7F7F7F7Fu) + 0x7F7F7F7Fu) | x) | 0x7F7F7F7Fu));
                }
            }
        } else {
            for (uint64_t i = a; i < b; ++i) k += text[i] == '\n';
        }
        if (n_fstart)  // breaks at bytes i in [a, b) in front of a file start i + 1
            for (uint32_t j = lower_bound_u32(fstart, n_fstart, (uint32_t)a + 1); j < n_fstart && fstart[j] <= b; ++j)
                k += text[fstart[j] - 1] != '\n';
        counts[c] = k;
    }
}

__global__ void ingest_newline_positions_kernel(uint64_t n_bytes, const char* __restrict__ text, const uint32_t* __restrict__ rank,
                                                uint32_t* __restrict__ nl_pos, const uint32_t* __restrict__ fstart, uint32_t n_fstart) {
    const uint64_t n_chunks = (n_bytes + INGEST_CHUNK - 1) / INGEST_CHUNK;
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t c = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; c < n_chunks; c += stride) {
        const uint64_t a = c * INGEST_CHUNK, b = min(a + INGEST_CHUNK, n_bytes);
        uint32_t r = rank[c];
        uint32_t j = n_fstart ? lower_bound_u32(fstart, n_fstart, (uint32_t)a + 1) : 0;
        for (uint64_t i = a; i < b; ++i) {
            const bool at_file_start = j < n_fstart && fstart[j] == i + 1;
            if (at_file_start) ++j;
            if (text[i] == '\n' || at_file_start) nl_pos[r++] = (uint32_t)i;
        }
    }
}

__device__ __forceinline__ bool is_digit(char c) { return c >= '0' && c <= '9'; }

// str::parse::<u32>(): optional '+', at least one digit, digits only, no overflow
__device__ bool parse_u32_field(const char* __restrict__ t, uint32_t a, uint32_t b, uint32_t& out) {
    if (a < b && t[a] == '+') ++a;
    if (a >= b) return false;
    unsigned long long v = 0;
    for (uint32_t i = a; i < b; ++i) {
        const char c = t[i];
        if (!is_digit(c)) return false;
        v = v * 10 + (unsigned long long)(c - '0');
        if (v > 0xFFFFFFFFull) return false;
    }
    out = (uint32_t)v;
    return true;
}

__device__ bool has_prefix(const char* __restrict__ t, uint32_t a, uint32_t b, const char* p, uint32_t n) {
    if (b - a < n) return false;
    for (uint32_t i = 0; i < n; ++i)
        if (t[a + i] != p[i]) return false;
    return true;
}

// The columns a line kernel writes per line of its window (keep = the line is kept), and the compaction writes per kept line.
// h / bo / bl: the line's key (FNV-1a hash, never 0; byte offset and length in the window), null for a format without keys.
struct LineCols {
    uint32_t *keep, *chr, *start, *end;
    unsigned long long* h;
    uint32_t *bo, *bl;
};

// status per line: 0 = skipped (comment / header), 1 = region, 2 = malformed.
// FILES (a text of several BED files back to back, files.file_offsets in bytes of the whole text): a file start is a line start
// even without a '\n' in front of it (the newline passes put a break there), the header rule applies to the first line of every
// file, chromosome names are not looked up but carried as the line's key for the caller's name discovery, and chr[li] receives
// the line's file index.  files.first_line[f] gets the text-wide index of file f's first line.
template <bool FILES>
__global__ void ingest_parse_lines_kernel(uint32_t n_lines, uint32_t n_newlines, uint64_t n_bytes, const char* __restrict__ text,
                                          const uint32_t* __restrict__ nl_pos, NameTable names, LineCols o,
                                          uint32_t* __restrict__ first_bad_line, BedFilesView files) {
    const uint32_t stride = gridDim.x * blockDim.x;
    for (uint32_t li = blockIdx.x * blockDim.x + threadIdx.x; li < n_lines; li += stride) {
        uint32_t a = li ? nl_pos[li - 1] + 1 : 0;
        uint32_t b = li < n_newlines ? nl_pos[li] : (uint32_t)n_bytes;
        bool nl_end = li < n_newlines;
        if (FILES && nl_end && text[b] != '\n') {  // a break in front of a file start: the line ends with its file
            ++b;
            nl_end = false;
        }
        // BufRead::lines strips "\n" and a "\r" right before it; a final line WITHOUT a newline keeps its '\r' (the reference then
        // fails to parse the field, and so do we)
        if (nl_end && b > a && text[b - 1] == '\r') --b;
        uint32_t k = 0, c = GTGPU_UNKNOWN_CHROM, s = 0, e = 0;
        bool first = li == 0;
        if (FILES) {  // the line's file: the last one that starts at or before it (empty files start where the next one does)
            const unsigned long long pos = files.byte0 + a;
            uint64_t lo = 0, hi = files.n_files;
            while (hi - lo > 1) {
                const uint64_t mid = (lo + hi) >> 1;
                if (files.file_offsets[mid] <= pos) lo = mid;
                else hi = mid;
            }
            c = (uint32_t)lo;
            first = files.file_offsets[lo] == pos;
            if (first) files.first_line[lo] = files.line0 + li;
        }
        if (has_prefix(text, a, b, "browser", 7) || has_prefix(text, a, b, "track", 5) || has_prefix(text, a, b, "#", 1)) {
            k = 0;
        } else {
            // tab-separated fields 0, 1, 2
            uint32_t t1 = a;
            while (t1 < b && text[t1] != '\t') ++t1;
            uint32_t t2 = t1 < b ? t1 + 1 : b;
            while (t2 < b && text[t2] != '\t') ++t2;
            uint32_t t3 = t2 < b ? t2 + 1 : b;
            while (t3 < b && text[t3] != '\t') ++t3;
            const bool three = t1 < b && t2 < b;  // at least two tabs = three parts
            const bool s_ok = three && parse_u32_field(text, t1 + 1, t2, s);
            if (first && three && !s_ok) {
                k = 0;  // a column-header first row without '#' (region_set.rs:118-131)
            } else if (!s_ok || !parse_u32_field(text, t2 + 1, t3, e)) {
                k = 2;
            } else {
                k = 1;
                const unsigned long long h = fnv1a64(text + a, t1 - a);
                if (FILES) {
                    o.h[li] = h ? h : 1;  // 0 marks an empty slot of the key table
                    o.bo[li] = a;
                    o.bl[li] = t1 - a;
                } else {
                    c = names.lookup(h, text + a, t1 - a);
                }
            }
        }
        if (k == 2) atomicMin(first_bad_line, li);
        o.keep[li] = k == 1;
        o.chr[li] = c;
        o.start[li] = s;
        o.end[li] = e;
    }
}

__device__ __forceinline__ uint32_t rank_of(const uint32_t* __restrict__ name_rank, uint32_t n_names, uint32_t c) {
    return c < n_names ? name_rank[c] : n_names;  // unknown names after every known one
}

// The record kernels of the sort loop with 64-bit indices: a batch of files may hold up to 2^32 - 2 records, and a 32-bit
// grid-stride index would wrap there.
// file (optional): the records' file indices, grouped; a pair that straddles two files is in order whatever its keys
__global__ void ingest_check_sorted_kernel(uint32_t n, const uint32_t* __restrict__ chr, const uint32_t* __restrict__ start,
                                           const uint32_t* __restrict__ name_rank, uint32_t n_names, uint32_t* __restrict__ unsorted,
                                           const uint32_t* __restrict__ file = nullptr) {
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i + 1 < n; i += stride) {
        if (file && file[i] != file[i + 1]) continue;
        const uint32_t ra = rank_of(name_rank, n_names, chr[i]), rb = rank_of(name_rank, n_names, chr[i + 1]);
        if (ra > rb || (ra == rb && start[i] > start[i + 1])) *unsorted = 1;
    }
}

__global__ void ingest_iota_kernel(uint32_t n, uint32_t* __restrict__ out) {
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) out[i] = (uint32_t)i;
}

// file (optional): the record's file index goes above the rank's rank_bits, so one pass orders by (file, rank)
__global__ void ingest_rank_keys_kernel(uint32_t n, const uint32_t* __restrict__ order, const uint32_t* __restrict__ chr,
                                        const uint32_t* __restrict__ name_rank, uint32_t n_names, uint32_t* __restrict__ keys,
                                        const uint32_t* __restrict__ file = nullptr, int rank_bits = 0) {
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        const uint32_t j = order[i];
        keys[i] = rank_of(name_rank, n_names, chr[j]) | (file ? file[j] << rank_bits : 0u);
    }
}

__global__ void ingest_gather_kernel(uint32_t n, const uint32_t* __restrict__ order, const uint32_t* __restrict__ chr,
                                     const uint32_t* __restrict__ start, const uint32_t* __restrict__ end, uint32_t* __restrict__ o_chr,
                                     uint32_t* __restrict__ o_start, uint32_t* __restrict__ o_end) {
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        const uint32_t j = order[i];
        o_chr[i] = chr[j];
        o_start[i] = start[j];
        o_end[i] = end[j];
    }
}

// ---- fragment files (gtars-tokenizers/src/utils/fragments.rs:12-82) ---------------------------------------------------------
__device__ __forceinline__ bool is_space(char c) { return c == ' ' || (c >= '\t' && c <= '\r'); }  // ASCII White_Space

// One thread per line: '#' lines are skipped; split_whitespace must give at least 5 fields (chr start end barcode ...),
// start and end parse as u32 — and with SUPPORT the fifth field too (Fragment::from_str, gtars-core/src/models/fragments.rs:16-44,
// which gtars-scoring reads through).  With BARCODE the barcode is carried as (FNV-1a hash, byte span); the count-matrix
// parse has no use for it and skips the hashing.
template <bool SUPPORT, bool BARCODE>
__global__ void ingest_parse_fragments_kernel(uint32_t n_lines, uint32_t n_newlines, uint64_t n_bytes, const char* __restrict__ text,
                                              const uint32_t* __restrict__ nl_pos, NameTable names, LineCols o,
                                              uint32_t* __restrict__ first_bad_line) {
    const uint32_t stride = gridDim.x * blockDim.x;
    for (uint32_t li = blockIdx.x * blockDim.x + threadIdx.x; li < n_lines; li += stride) {
        uint32_t a = li ? nl_pos[li - 1] + 1 : 0;
        uint32_t b = li < n_newlines ? nl_pos[li] : (uint32_t)n_bytes;
        if (li < n_newlines && b > a && text[b - 1] == '\r') --b;  // only a '\r' in front of a '\n' is part of the line ending
        uint32_t k = 0, c = GTGPU_UNKNOWN_CHROM, s = 0, e = 0, bo = 0, bl = 0, sup = 0;
        unsigned long long h = 1;
        if (!(b > a && text[a] == '#')) {
            uint32_t fa[5], fb[5], nf = 0, p = a;
            while (nf < 5) {
                while (p < b && is_space(text[p])) ++p;
                if (p >= b) break;
                fa[nf] = p;
                while (p < b && !is_space(text[p])) ++p;
                fb[nf++] = p;
            }
            if (nf < 5 || !parse_u32_field(text, fa[1], fb[1], s) || !parse_u32_field(text, fa[2], fb[2], e) ||
                (SUPPORT && !parse_u32_field(text, fa[4], fb[4], sup))) {
                k = 2;
            } else {
                k = 1;
                c = names.lookup(fnv1a64(text + fa[0], fb[0] - fa[0]), text + fa[0], fb[0] - fa[0]);
                if (BARCODE) {
                    bo = fa[3];
                    bl = fb[3] - fa[3];
                    h = fnv1a64(text + bo, bl);
                    if (h == 0) h = 1;  // 0 marks an empty slot of the key table
                }
            }
        }
        if (k == 2) atomicMin(first_bad_line, li);
        o.keep[li] = k == 1;
        o.chr[li] = c;
        o.start[li] = s;
        o.end[li] = e;
        if (BARCODE) {
            o.h[li] = h;
            o.bo[li] = bo;
            o.bl[li] = bl;
        }
    }
}

__global__ void ingest_compact_lines_kernel(uint32_t n_lines, const uint32_t* __restrict__ pos, LineCols p, LineCols o) {
    const uint32_t stride = gridDim.x * blockDim.x;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n_lines; i += stride)
        if (p.keep[i]) {
            const uint32_t q = pos[i];
            o.chr[q] = p.chr[i];
            o.start[q] = p.start[i];
            o.end[q] = p.end[i];
            if (o.h) {  // uniform per launch: only some formats carry keys
                o.h[q] = p.h[i];
                o.bo[q] = p.bo[i];
                o.bl[q] = p.bl[i];
            }
        }
}

// ---- the key table (KeyTable): open addressing on the 64-bit key hash, one table over all windows of a text -------------------
// A window's lines are numbered text-wide (base + k), so a slot's first-appearance index is the text-wide index of the key's
// first line.  Per line the table keeps that index (id); per slot the key's byte length, its offset in the arena (the window
// that first sees a key copies its bytes there, because the text of a plain-text window leaves the device with it), "seen on
// a chromosome of the name table" (known, when not every key is kept) and, when asked for, its first byte offset in the text.
struct KeySlots {
    unsigned long long *hash, *soff, *first_byte;
    uint32_t *first, *klen, *known;
};

__device__ __forceinline__ uint32_t key_home(unsigned long long key, uint32_t mask) {
    return (uint32_t)((key * 0x9E3779B97F4A7C15ull) >> 32) & mask;
}

// every line finds or claims its key's slot (slot_of[k]; mask + 1 when the table is full) and lowers the slot's first appearance
__global__ void ingest_key_insert_kernel(uint32_t n, const unsigned long long* __restrict__ h, uint32_t mask, unsigned long long* hash,
                                         uint32_t* first, uint32_t* __restrict__ slot_of, uint32_t base, uint32_t* __restrict__ full) {
    const uint32_t stride = gridDim.x * blockDim.x;
    for (uint32_t k = blockIdx.x * blockDim.x + threadIdx.x; k < n; k += stride) {
        const unsigned long long key = h[k];
        uint32_t slot = key_home(key, mask), probes = 0;
        for (;;) {
            unsigned long long prev = hash[slot];  // a set key never changes: only an empty slot needs the CAS
            if (prev == 0ull) prev = atomicCAS(hash + slot, 0ull, key);
            if (prev == 0ull || prev == key) break;
            slot = (slot + 1) & mask;
            if (++probes > mask) {  // more keys than slots: reported, never spun on
                atomicOr(full, 1u);
                slot = mask + 1;
                break;
            }
        }
        // consecutive lines often share a key: the first lane of each group of equal slots lowers the first appearance
        const unsigned same = __match_any_sync(__activemask(), slot);
        if (slot <= mask && (threadIdx.x & 31) == (unsigned)(__ffs(same) - 1) && first[slot] > base + k) atomicMin(first + slot, base + k);
        slot_of[k] = slot;
    }
}

__global__ void ingest_key_rehash_kernel(uint64_t old_cap, KeySlots o, uint32_t mask, KeySlots t) {
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t s = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; s < old_cap; s += stride) {
        const unsigned long long key = o.hash[s];
        if (!key) continue;
        uint32_t slot = key_home(key, mask);
        while (atomicCAS(t.hash + slot, 0ull, key) != 0ull) slot = (slot + 1) & mask;  // keys are distinct
        t.first[slot] = o.first[s];
        t.soff[slot] = o.soff[s];
        t.klen[slot] = o.klen[s];
        if (t.known) t.known[slot] = o.known[s];
        if (t.first_byte) t.first_byte[slot] = o.first_byte[s];
    }
}

// per line its key's first appearance; per key first seen in this window its length (wlen, 0 for other lines, for the arena
// scan); known keys are marked; n_new counts the keys first seen here
__global__ void ingest_key_heads_kernel(uint32_t n, uint32_t base, const uint32_t* __restrict__ slot_of, const uint32_t* __restrict__ first,
                                        const uint32_t* __restrict__ chr, const uint32_t* __restrict__ bl, uint32_t n_names, uint32_t mask,
                                        uint32_t* __restrict__ id, uint32_t* __restrict__ klen, uint32_t* __restrict__ known,
                                        uint32_t* __restrict__ wlen, uint32_t* __restrict__ n_new) {
    const uint32_t stride = gridDim.x * blockDim.x;
    for (uint32_t k = blockIdx.x * blockDim.x + threadIdx.x; k < n; k += stride) {
        const uint32_t s = slot_of[k], g = base + k;
        const bool in_table = s <= mask;  // the lines of a full table are reported by the insert and skipped here
        const uint32_t f = in_table ? first[s] : 0xFFFFFFFFu;
        const bool head = f == g;
        id[g] = f;
        wlen[k] = head ? bl[k] : 0u;
        if (head) klen[s] = bl[k];
        if (known && in_table && chr[k] < n_names) known[s] = 1u;  // files.rs:106-129: a consensus chromosome creates the barcode's entry
        const unsigned m = __ballot_sync(__activemask(), head);
        if (head && (threadIdx.x & 31) == (unsigned)(__ffs(m) - 1)) atomicAdd(n_new, (uint32_t)__popc(m));
    }
}

__global__ void ingest_key_claim_kernel(uint32_t n, uint32_t base, const char* __restrict__ text, const uint32_t* __restrict__ slot_of,
                                        const uint32_t* __restrict__ id, const uint32_t* __restrict__ bo, const uint32_t* __restrict__ bl,
                                        const uint32_t* __restrict__ wpos, uint64_t used, char* __restrict__ arena,
                                        unsigned long long* __restrict__ soff, uint64_t byte0, unsigned long long* __restrict__ first_byte) {
    const uint32_t stride = gridDim.x * blockDim.x;
    for (uint32_t k = blockIdx.x * blockDim.x + threadIdx.x; k < n; k += stride) {
        if (id[base + k] != base + k) continue;
        const uint64_t p = used + wpos[k];
        for (uint32_t i = 0; i < bl[k]; ++i) arena[p + i] = text[bo[k] + i];
        soff[slot_of[k]] = p;
        if (first_byte) first_byte[slot_of[k]] = byte0 + bo[k];
    }
}

// every later line of a key has its first appearance's bytes (a 64-bit hash collision would merge two keys)
__global__ void ingest_key_check_kernel(uint32_t n, uint32_t base, const char* __restrict__ text, const uint32_t* __restrict__ slot_of,
                                        const uint32_t* __restrict__ id, const uint32_t* __restrict__ bo, const uint32_t* __restrict__ bl,
                                        const uint32_t* __restrict__ klen, const char* __restrict__ arena,
                                        const unsigned long long* __restrict__ soff, uint32_t* __restrict__ collision) {
    const uint32_t stride = gridDim.x * blockDim.x;
    for (uint32_t k = blockIdx.x * blockDim.x + threadIdx.x; k < n; k += stride) {
        if (id[base + k] == base + k) continue;
        const uint32_t s = slot_of[k];
        const uint64_t p = soff[s];
        bool same = klen[s] == bl[k];
        for (uint32_t i = 0; same && i < bl[k]; ++i) same = arena[p + i] == text[bo[k] + i];
        if (!same) *collision = 1;
    }
}

// after the last window: the first appearance and slot of every kept key (keep_all <=> known == nullptr), in no particular order
__global__ void ingest_key_kept_kernel(uint64_t cap, const unsigned long long* __restrict__ hash, const uint32_t* __restrict__ first,
                                       const uint32_t* __restrict__ known, uint32_t* __restrict__ kfirst, uint32_t* __restrict__ kslot,
                                       uint32_t* __restrict__ n_kept) {
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t s = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; s < cap; s += stride) {
        const bool kp = hash[s] && (!known || known[s]);
        const unsigned act = __activemask(), m = __ballot_sync(act, kp);
        if (!m) continue;  // uniform over the active lanes
        const int lane = threadIdx.x & 31, leader = __ffs(m) - 1;
        uint32_t at = 0;
        if (lane == leader) at = atomicAdd(n_kept, (uint32_t)__popc(m));
        at = __shfl_sync(act, at, leader) + __popc(m & ((1u << lane) - 1));
        if (kp) {
            kfirst[at] = first[s];
            kslot[at] = (uint32_t)s;
        }
    }
}

// kept key i (first-appearance order): its name's length (for the offset scan), or its (first byte, length) span
__global__ void ingest_key_lengths_kernel(uint32_t n_kept, const uint32_t* __restrict__ kslot, const uint32_t* __restrict__ klen,
                                          const unsigned long long* __restrict__ first_byte, unsigned long long* __restrict__ len,
                                          uint32_t* __restrict__ spans) {
    const uint32_t stride = gridDim.x * blockDim.x;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n_kept; i += stride) {
        const uint32_t s = kslot[i];
        if (len) len[i] = klen[s];
        if (spans) {
            spans[2 * (uint64_t)i] = (uint32_t)first_byte[s];
            spans[2 * (uint64_t)i + 1] = klen[s];
        }
    }
}

__global__ void ingest_key_names_kernel(uint32_t n_kept, const uint32_t* __restrict__ kslot, const uint32_t* __restrict__ klen,
                                        const unsigned long long* __restrict__ soff, const char* __restrict__ arena,
                                        const unsigned long long* __restrict__ name_off, char* __restrict__ blob) {
    const uint32_t stride = gridDim.x * blockDim.x;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n_kept; i += stride) {
        const uint32_t s = kslot[i];
        for (uint32_t j = 0; j < klen[s]; ++j) blob[name_off[i] + j] = arena[soff[s] + j];
    }
}

// a line's first-appearance index -> its key's dense id: the index's position among the kept keys' sorted first appearances.
// A line of a dropped key lies on an unknown chromosome (it has no hit), so any valid id serves it.
__global__ void ingest_key_ids_kernel(uint64_t n, const uint32_t* __restrict__ kfirst, uint32_t n_kept, uint32_t* __restrict__ id) {
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t g = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; g < n; g += stride) {
        const uint32_t f = id[g], i = lower_bound_u32(kfirst, n_kept, f);
        id[g] = i < n_kept && kfirst[i] == f ? i : 0u;
    }
}

// Name table in scratch SC_SET_ID: FNV-1a hashes of the caller's chromosome names, sorted for the device lookup, and (with_rank)
// the names' lexicographic ranks for the sort of gtgpu_parse_bed.
int32_t upload_name_table(gtgpu_ctx* ctx, uint32_t n_names, const char* names, const uint32_t* name_offsets, NameTable* out,
                          bool with_rank) {
    cudaStream_t st = ctx->stream;
    std::vector<unsigned long long> hash(n_names), hash_sorted(n_names);
    std::vector<uint32_t> hash_id(n_names), rank(with_rank ? n_names : 0);
    for (uint32_t i = 0; i < n_names; ++i) hash[i] = fnv1a64(names + name_offsets[i], name_offsets[i + 1] - name_offsets[i]);
    std::iota(hash_id.begin(), hash_id.end(), 0u);
    std::sort(hash_id.begin(), hash_id.end(), [&](uint32_t a, uint32_t b) { return hash[a] != hash[b] ? hash[a] < hash[b] : a < b; });
    for (uint32_t i = 0; i < n_names; ++i) hash_sorted[i] = hash[hash_id[i]];
    if (with_rank) {
        std::vector<uint32_t> by_name(n_names);
        std::iota(by_name.begin(), by_name.end(), 0u);
        auto name_of = [&](uint32_t i) { return std::string(names + name_offsets[i], names + name_offsets[i + 1]); };
        std::stable_sort(by_name.begin(), by_name.end(), [&](uint32_t a, uint32_t b) { return name_of(a) < name_of(b); });
        for (uint32_t r = 0; r < n_names; ++r) rank[by_name[r]] = r;  // equal strings cannot occur in a name table
    }
    const uint32_t blob_bytes = n_names ? name_offsets[n_names] : 0;
    char* d_names;
    GT_TRY(ctx->scratch_get(SC_SET_ID, (size_t)n_names * 16 + ((size_t)n_names + 1) * 4 + blob_bytes + 64, (void**)&d_names));
    // layout: hashes (8-byte aligned first), offsets, hash ids, ranks, blob
    unsigned long long* d_hash = reinterpret_cast<unsigned long long*>(d_names);
    uint32_t* d_noff = reinterpret_cast<uint32_t*>(d_hash + n_names);
    uint32_t* d_hid = d_noff + n_names + 1;
    uint32_t* d_rank = d_hid + n_names;
    char* d_blob = reinterpret_cast<char*>(d_rank + n_names);
    if (n_names) {
        GT_CUDA(cudaMemcpyAsync(d_hash, hash_sorted.data(), (size_t)n_names * 8, cudaMemcpyHostToDevice, st));
        GT_CUDA(cudaMemcpyAsync(d_hid, hash_id.data(), (size_t)n_names * 4, cudaMemcpyHostToDevice, st));
        if (with_rank) GT_CUDA(cudaMemcpyAsync(d_rank, rank.data(), (size_t)n_names * 4, cudaMemcpyHostToDevice, st));
        if (blob_bytes) GT_CUDA(cudaMemcpyAsync(d_blob, names, blob_bytes, cudaMemcpyHostToDevice, st));
    }
    GT_CUDA(cudaMemcpyAsync(d_noff, name_offsets ? name_offsets : (const uint32_t*)&blob_bytes, ((size_t)n_names + 1) * 4,
                            cudaMemcpyHostToDevice, st));
    GT_CUDA(cudaStreamSynchronize(st));  // the host vectors above are pageable and go out of scope
    *out = NameTable{d_blob, d_noff, d_hash, d_hid, n_names, with_rank ? d_rank : nullptr};
    return GTGPU_OK;
}

// Line breaks of device text (every '\n', and the breaks in front of the d_fstart file starts): *d_nl (scratch SC_IN3_END) gets
// the n_breaks break positions, *n_lines counts the lines (the last one may end without a break).  Synchronises the ctx stream.
static int32_t line_breaks_locked(gtgpu_ctx* ctx, const char* d_text, uint64_t n_bytes, const uint32_t* d_fstart, uint32_t n_fstart,
                                  uint32_t* n_breaks, uint32_t* n_lines, uint32_t** d_nl) {
    cudaStream_t st = ctx->stream;
    uint32_t *d_counts, *d_crank;
    void* d_tmp;
    const uint64_t n_chunks = (n_bytes + INGEST_CHUNK - 1) / INGEST_CHUNK;
    GT_TRY(ctx->scratch_get(SC_COUNTS, n_chunks * 4 + 4, (void**)&d_counts));
    GT_TRY(ctx->scratch_get(SC_IN3_CHR, n_chunks * 4 + 4, (void**)&d_crank));
    GT_TRY(ctx->scratch_get(SC_IN3_START, exclusive_scan_temp_bytes(n_chunks, 4), &d_tmp));
    ingest_count_newlines_kernel<<<grid_for(ctx, n_chunks), 256, 0, st>>>(n_bytes, d_text, d_counts, d_fstart, n_fstart);
    ctx->launches++;
    GT_TRY(exclusive_scan<uint32_t>(ctx, d_counts, d_crank, n_chunks, d_tmp));
    uint32_t last[2];
    GT_CUDA(cudaMemcpyAsync(&last[0], d_crank + n_chunks - 1, 4, cudaMemcpyDeviceToHost, st));
    GT_CUDA(cudaMemcpyAsync(&last[1], d_counts + n_chunks - 1, 4, cudaMemcpyDeviceToHost, st));
    char last_byte = 0;  // read back from the device: with device-resident text there is no host copy
    GT_CUDA(cudaMemcpyAsync(&last_byte, d_text + n_bytes - 1, 1, cudaMemcpyDeviceToHost, st));
    GT_CUDA(cudaStreamSynchronize(st));
    *n_breaks = last[0] + last[1];
    *n_lines = *n_breaks + (last_byte != '\n' ? 1u : 0u);
    GT_TRY(ctx->scratch_get(SC_IN3_END, (size_t)*n_breaks * 4 + 4, (void**)d_nl));
    ingest_newline_positions_kernel<<<grid_for(ctx, n_chunks), 256, 0, st>>>(n_bytes, d_text, d_crank, *d_nl, d_fstart, n_fstart);
    ctx->launches++;
    return GTGPU_OK;
}

// The line front end of every device text parser: line breaks, the format's line kernel, compaction of the kept lines.
int32_t parse_lines_locked(gtgpu_ctx* ctx, const char* d_text, uint64_t n_bytes, LineFormat fmt, const NameTable& nt,
                           const BedFilesView& files, ParsedLines* out) {
    cudaStream_t st = ctx->stream;
    uint32_t *d_nl, *d_pos;
    void* d_tmp;
    uint64_t* d_misc;
    uint32_t n_breaks = 0, n_lines = 0;
    GT_TRY(line_breaks_locked(ctx, d_text, n_bytes, files.fstart, files.n_fstart, &n_breaks, &n_lines, &d_nl));
    const bool keys = fmt == BED_FILE_LINES || fmt == FRAG_TOKENIZE || fmt == FRAG_SCORE_BARCODES;
    const size_t lb = (size_t)n_lines * 4 + 8;
    LineCols p{}, o{};  // per line, per kept line
    GT_TRY(ctx->scratch_get(SC_IN3_START, exclusive_scan_temp_bytes(n_lines, 4), &d_tmp));
    GT_TRY(ctx->scratch_get(SC_ING_0, lb, (void**)&p.keep));
    GT_TRY(ctx->scratch_get(SC_ING_1, lb, (void**)&d_pos));
    GT_TRY(ctx->scratch_get(SC_IN2_CHR, lb, (void**)&p.chr));
    GT_TRY(ctx->scratch_get(SC_IN2_START, lb, (void**)&p.start));
    GT_TRY(ctx->scratch_get(SC_IN2_END, lb, (void**)&p.end));
    GT_TRY(ctx->scratch_get(SC_CHR, lb, (void**)&o.chr));
    GT_TRY(ctx->scratch_get(SC_START, lb, (void**)&o.start));
    GT_TRY(ctx->scratch_get(SC_END, lb, (void**)&o.end));
    if (keys) {
        GT_TRY(ctx->scratch_get(SC_ING_2, lb * 2, (void**)&p.h));
        GT_TRY(ctx->scratch_get(SC_ING_3, lb, (void**)&p.bo));
        GT_TRY(ctx->scratch_get(SC_ING_4, lb, (void**)&p.bl));
        GT_TRY(ctx->scratch_get(SC_ING_5, lb * 2, (void**)&o.h));
        GT_TRY(ctx->scratch_get(SC_ING_6, lb, (void**)&o.bo));
        GT_TRY(ctx->scratch_get(SC_ING_7, lb, (void**)&o.bl));
    }
    GT_TRY(ctx->scratch_get(SC_MISC, 64, (void**)&d_misc));
    uint32_t* d_flags = reinterpret_cast<uint32_t*>(d_misc);  // [0] first malformed line, [1..3] for the caller
    const uint32_t init[4] = {0xFFFFFFFFu, 0u, 0u, 0u};
    GT_CUDA(cudaMemcpyAsync(d_flags, init, 16, cudaMemcpyHostToDevice, st));
    const int grid = grid_for(ctx, n_lines);
    switch (fmt) {
    case BED_LINES:
        ingest_parse_lines_kernel<false><<<grid, 256, 0, st>>>(n_lines, n_breaks, n_bytes, d_text, d_nl, nt, p, d_flags, files);
        break;
    case BED_FILE_LINES:
        ingest_parse_lines_kernel<true><<<grid, 256, 0, st>>>(n_lines, n_breaks, n_bytes, d_text, d_nl, nt, p, d_flags, files);
        break;
    case FRAG_TOKENIZE:
        ingest_parse_fragments_kernel<false, true><<<grid, 256, 0, st>>>(n_lines, n_breaks, n_bytes, d_text, d_nl, nt, p, d_flags);
        break;
    case FRAG_SCORE_MATRIX:
        ingest_parse_fragments_kernel<true, false><<<grid, 256, 0, st>>>(n_lines, n_breaks, n_bytes, d_text, d_nl, nt, p, d_flags);
        break;
    case FRAG_SCORE_BARCODES:
        ingest_parse_fragments_kernel<true, true><<<grid, 256, 0, st>>>(n_lines, n_breaks, n_bytes, d_text, d_nl, nt, p, d_flags);
        break;
    }
    ctx->launches++;
    GT_TRY(exclusive_scan<uint32_t>(ctx, p.keep, d_pos, n_lines, d_tmp));
    ingest_compact_lines_kernel<<<grid, 256, 0, st>>>(n_lines, d_pos, p, o);
    ctx->launches++;
    uint32_t tail[2], flags[1];
    GT_CUDA(cudaMemcpyAsync(&tail[0], d_pos + n_lines - 1, 4, cudaMemcpyDeviceToHost, st));
    GT_CUDA(cudaMemcpyAsync(&tail[1], p.keep + n_lines - 1, 4, cudaMemcpyDeviceToHost, st));
    GT_CUDA(cudaMemcpyAsync(flags, d_flags, 4, cudaMemcpyDeviceToHost, st));
    GT_CUDA(cudaStreamSynchronize(st));
    *out = ParsedLines{};
    out->n_lines = n_lines;
    out->bad_line = flags[0];
    out->n = flags[0] == 0xFFFFFFFFu ? tail[0] + tail[1] : 0;
    out->chr = o.chr;
    out->start = o.start;
    out->end = o.end;
    out->h = o.h;
    out->bo = o.bo;
    out->bl = o.bl;
    out->breaks = d_nl;
    uint32_t* const line_sized[5] = {p.keep, d_pos, p.chr, p.start, p.end};  // free again
    std::copy(line_sized, line_sized + 5, out->free);
    out->tmp = d_tmp;
    out->flags = d_flags;
    return GTGPU_OK;
}

// ---- fragment text of any size, window by window (scoring and tokenization) --------------------------------------------------
// The text is parsed in windows (the parse kernels address a window with u32 positions): a window ends right after the first
// '\n' at or past its nominal size, so it holds whole lines, and a window's local line index plus the lines of the windows
// before it is the file-wide index the host parser reports.  Plain text is copied window by window (the copy of window k+1,
// through pinned staging on the copy stream, overlaps the kernels of window k); device text (e.g. inflated gzip members) is
// read where it is.

// GTGPU_INGEST_WINDOW=<bytes>, read per call: nominal window size (results never depend on it)
static uint64_t ingest_window_bytes() {
    uint64_t w = 2ull << 30;
    if (const char* env = getenv("GTGPU_INGEST_WINDOW")) {
        const uint64_t v = strtoull(env, nullptr, 10);
        if (v) w = v;
    }
    return std::min<uint64_t>(w, 3ull << 30);
}

struct StagingScope {  // pinned staging blocks and their events, returned to the ctx when the call ends
    gtgpu_ctx* ctx;
    PinnedBlock pin[2];
    cudaEvent_t ev[2] = {nullptr, nullptr};
    bool used[2] = {false, false};
    explicit StagingScope(gtgpu_ctx* c) : ctx(c) {}
    ~StagingScope() {
        cudaStreamSynchronize(ctx->copy_in);
        for (int b = 0; b < 2; ++b) {
            if (ev[b]) cudaEventDestroy(ev[b]);
            ctx->pinned_put(pin[b]);
        }
    }
};

int32_t for_each_window(gtgpu_ctx* ctx, const Text& t, const std::string& who, const WindowFn& fn) {
    cudaStream_t st = ctx->stream;
    const uint64_t n_bytes = t.n_bytes;
    const char *host_text = t.on_device ? nullptr : t.bytes, *dev_text = t.on_device ? t.bytes : nullptr;
    const uint64_t W = ingest_window_bytes();
    std::vector<uint64_t> cut{0};  // window w = [cut[w], cut[w + 1])
    while (cut.back() < n_bytes) {
        const uint64_t a = cut.back();
        uint64_t b = n_bytes;
        if (n_bytes - a > W) {
            const uint64_t p = a + W - 1;
            if (host_text) {
                const void* q = memchr(host_text + p, '\n', n_bytes - p);
                if (q) b = (uint64_t)((const char*)q - host_text) + 1;
            } else {
                char piece[4096];
                for (uint64_t q = p; q < n_bytes && b == n_bytes; q += sizeof piece) {
                    const uint64_t len = std::min<uint64_t>(sizeof piece, n_bytes - q);
                    GT_CUDA(cudaMemcpyAsync(piece, dev_text + q, len, cudaMemcpyDeviceToHost, st));
                    GT_CUDA(cudaStreamSynchronize(st));
                    const void* nl = memchr(piece, '\n', len);
                    if (nl) b = q + (uint64_t)((const char*)nl - piece) + 1;
                }
            }
        }
        if (b - a >= 0xFFFFFFF0ull) return fail(GTGPU_ERR_UNSUPPORTED, who + ": a line of 4 GiB or more");
        cut.push_back(b);
    }
    const size_t n_win = cut.size() - 1;
    uint64_t max_win = 0;
    for (size_t w = 0; w < n_win; ++w) max_win = std::max(max_win, cut[w + 1] - cut[w]);
    uint64_t first_line = 0;
    uint32_t n_lines = 0;
    if (dev_text) {
        char* d_copy = nullptr;  // windows that do not start 16-byte aligned are moved to aligned scratch (the newline scan loads 16 B)
        for (size_t w = 0; w < n_win; ++w) {
            const char* d = dev_text + cut[w];
            if (reinterpret_cast<uintptr_t>(d) & 15) {
                if (!d_copy) GT_TRY(ctx->scratch_get(SC_WIN_A, max_win + 64, (void**)&d_copy));
                GT_CUDA(cudaMemcpyAsync(d_copy, d, cut[w + 1] - cut[w], cudaMemcpyDeviceToDevice, st));
                d = d_copy;
            }
            GT_TRY(fn(d, cut[w + 1] - cut[w], cut[w], first_line, &n_lines));
            first_line += n_lines;
        }
        return GTGPU_OK;
    }
    char* dbuf[2] = {nullptr, nullptr};
    GT_TRY(ctx->scratch_get(SC_WIN_A, max_win + 64, (void**)&dbuf[0]));
    if (n_win > 1) GT_TRY(ctx->scratch_get(SC_WIN_B, max_win + 64, (void**)&dbuf[1]));
    StagingScope sg(ctx);
    const uint64_t piece = std::min<uint64_t>(max_win, 64ull << 20);
    for (int b = 0; b < 2; ++b) {
        GT_TRY(ctx->pinned_get(piece, &sg.pin[b]));
        GT_CUDA(cudaEventCreateWithFlags(&sg.ev[b], cudaEventDisableTiming));
    }
    // window w -> dbuf[w % 2] through the two pinned pieces; runs on a helper thread while the kernels of window w - 1 run
    std::string stage_err;
    auto stage = [&](size_t w) -> int32_t {
        if (cudaSetDevice(ctx->device) != cudaSuccess) return GTGPU_ERR_CUDA;
        cudaError_t e = cudaSuccess;
        uint64_t j = 0;
        for (uint64_t off = cut[w]; off < cut[w + 1] && e == cudaSuccess; off += piece, ++j) {
            const int b = (int)(j & 1);
            const uint64_t len = std::min(piece, cut[w + 1] - off);
            if (sg.used[b]) e = cudaEventSynchronize(sg.ev[b]);
            if (e != cudaSuccess) break;
            memcpy(sg.pin[b].ptr, host_text + off, len);
            e = cudaMemcpyAsync(dbuf[w & 1] + (off - cut[w]), sg.pin[b].ptr, len, cudaMemcpyHostToDevice, ctx->copy_in);
            if (e == cudaSuccess) e = cudaEventRecord(sg.ev[b], ctx->copy_in);
            sg.used[b] = true;
        }
        if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->copy_in);
        if (e != cudaSuccess) stage_err = std::string("H2D of the text: ") + cudaGetErrorString(e);
        return e == cudaSuccess ? GTGPU_OK : GTGPU_ERR_CUDA;
    };
    int32_t s_next = stage(0);
    for (size_t w = 0; w < n_win && s_next == GTGPU_OK; ++w) {
        std::thread helper;
        if (w + 1 < n_win) helper = std::thread([&, w] { s_next = stage(w + 1); });
        const int32_t s = fn(dbuf[w & 1], cut[w + 1] - cut[w], cut[w], first_line, &n_lines);
        if (helper.joinable()) helper.join();
        if (s != GTGPU_OK) return s;
        first_line += n_lines;
    }
    if (s_next != GTGPU_OK) return fail(s_next, who + ": " + stage_err);
    return GTGPU_OK;
}

// RegionSet::sort (region_set.rs:502-505) of n parsed records: stable by (chromosome rank, start), within each file when `file` (the
// records' file indices, in file order) is given.  When some pair is out of order: stable radix passes by start, then by rank (the
// file index folded above it when both fit 32 bits, else one more pass by file), and a gather.  The sorted columns replace *chr /
// *start / *end; they lie in scratch SC_ING_0..3, which the fused find after the sort does not touch.  The caller holds ctx->mu.
static int32_t sort_regions_locked(gtgpu_ctx* ctx, uint32_t n, const NameTable& nt, uint32_t n_names, const uint32_t* file,
                                   uint64_t n_files, const uint32_t** chr, const uint32_t** start, const uint32_t** end) {
    cudaStream_t st = ctx->stream;
    uint32_t* d_flag;
    GT_TRY(ctx->scratch_get(SC_MISC, 64, (void**)&d_flag));
    GT_CUDA(cudaMemsetAsync(d_flag, 0, 4, st));
    ingest_check_sorted_kernel<<<grid_for(ctx, n), 256, 0, st>>>(n, *chr, *start, nt.rank, n_names, d_flag, file);
    ctx->launches++;
    uint32_t unsorted = 0;
    GT_CUDA(cudaMemcpyAsync(&unsorted, d_flag, 4, cudaMemcpyDeviceToHost, st));
    GT_CUDA(cudaStreamSynchronize(st));
    GT_CUDA(cudaGetLastError());
    if (!unsorted) return GTGPU_OK;
    uint32_t *k_a, *v_a, *k_b, *v_b;
    void* d_tmp;
    GT_TRY(ctx->scratch_get(SC_ING_0, (size_t)n * 4, (void**)&k_a));
    GT_TRY(ctx->scratch_get(SC_ING_1, (size_t)n * 4, (void**)&v_a));
    GT_TRY(ctx->scratch_get(SC_ING_2, (size_t)n * 4, (void**)&k_b));
    GT_TRY(ctx->scratch_get(SC_ING_3, (size_t)n * 4, (void**)&v_b));
    GT_TRY(ctx->scratch_get(SC_IN3_START, radix_sort_temp_bytes(n), &d_tmp));
    GT_CUDA(cudaMemcpyAsync(k_a, *start, (size_t)n * 4, cudaMemcpyDeviceToDevice, st));
    ingest_iota_kernel<<<grid_for(ctx, n), 256, 0, st>>>(n, v_a);
    ctx->launches++;
    int in_b = 0;
    GT_TRY(radix_sort_pairs(ctx, n, k_a, v_a, k_b, v_b, 32, d_tmp, &in_b));
    if (in_b) { std::swap(k_a, k_b); std::swap(v_a, v_b); }
    const int rank_bits = bits_for_value(n_names), file_bits = file ? bits_for_value(n_files - 1) : 0;
    const bool fold = file && rank_bits + file_bits <= 32;
    ingest_rank_keys_kernel<<<grid_for(ctx, n), 256, 0, st>>>(n, v_a, *chr, nt.rank, n_names, k_a, fold ? file : nullptr, rank_bits);
    ctx->launches++;
    GT_TRY(radix_sort_pairs(ctx, n, k_a, v_a, k_b, v_b, fold ? rank_bits + file_bits : rank_bits, d_tmp, &in_b));
    if (in_b) { std::swap(k_a, k_b); std::swap(v_a, v_b); }
    if (file && !fold) {
        GT_TRY(launch_gather_u32(ctx, n, file, v_a, k_a));
        GT_TRY(radix_sort_pairs(ctx, n, k_a, v_a, k_b, v_b, file_bits, d_tmp, &in_b));
        if (in_b) { std::swap(k_a, k_b); std::swap(v_a, v_b); }
    }
    // the order is v_a; the other three buffers take the sorted columns
    ingest_gather_kernel<<<grid_for(ctx, n), 256, 0, st>>>(n, v_a, *chr, *start, *end, k_a, k_b, v_b);
    ctx->launches++;
    *chr = k_a;
    *start = k_b;
    *end = v_b;
    GT_CUDA(cudaGetLastError());
    return GTGPU_OK;
}

// Parses and sorts on the device.  On success *d_chr / *d_start / *d_end point at n_out regions in device scratch
// (valid until the next call on this ctx).  The caller holds ctx->mu.
static int32_t parse_bed_locked(gtgpu_ctx* ctx, const Text& t, uint32_t n_names, const char* names, const uint32_t* name_offsets,
                                uint64_t* n_out, const uint32_t** d_chr, const uint32_t** d_start, const uint32_t** d_end) {
    const uint64_t n_bytes = t.n_bytes;
    if (n_bytes >= 0xFFFFFFF0ull) return fail(GTGPU_ERR_UNSUPPORTED, "parse_bed: at most 4 GiB of text per call (split at a line boundary)");
    if (n_names >= 0x7FFFFFFFu) return fail(GTGPU_ERR_INVALID, "parse_bed: too many chromosome names");
    *n_out = 0;
    if (n_bytes == 0) return fail(GTGPU_ERR_INVALID, "parse_bed: EmptyRegionSet (no regions in the text)");

    const char* d_text = t.bytes;
    if (!t.on_device) {
        GT_TRY(ctx->scratch_get(SC_OUT_IDS2, n_bytes + 64, (void**)&d_text));
        GT_CUDA(cudaMemcpyAsync((char*)d_text, t.bytes, n_bytes, cudaMemcpyHostToDevice, ctx->stream));
    }
    NameTable nt;
    GT_TRY(upload_name_table(ctx, n_names, names, name_offsets, &nt, true));  // synchronises: the host's text may be reused after it
    ParsedLines pl;
    GT_TRY(parse_lines_locked(ctx, d_text, n_bytes, BED_LINES, nt, BedFilesView{}, &pl));
    if (pl.bad_line != 0xFFFFFFFFu)
        return fail(GTGPU_ERR_INVALID, "parse_bed: RegionParseError: cannot parse start / end position on line " + std::to_string((uint64_t)pl.bad_line + 1));
    if (pl.n == 0) return fail(GTGPU_ERR_INVALID, "parse_bed: EmptyRegionSet (no regions in the text)");
    *d_chr = pl.chr;
    *d_start = pl.start;
    *d_end = pl.end;
    GT_TRY(sort_regions_locked(ctx, pl.n, nt, n_names, nullptr, 0, d_chr, d_start, d_end));
    *n_out = pl.n;
    return GTGPU_OK;
}

int32_t DevMem::reserve(size_t bytes, size_t keep, cudaStream_t st) {
    if (cap >= bytes) return GTGPU_OK;
    void* p = nullptr;
    size_t want = std::max(bytes, cap + cap / 2);
    if (cudaMalloc(&p, want) != cudaSuccess) {
        cudaGetLastError();
        want = bytes;
        cudaError_t e = cudaMalloc(&p, want);
        if (e != cudaSuccess) return fail(GTGPU_ERR_NOMEM, "cudaMalloc(" + std::to_string(bytes) + " B): " + cudaGetErrorString(e));
    }
    if (keep) GT_CUDA(cudaMemcpyAsync(p, ptr, keep, cudaMemcpyDeviceToDevice, st));
    GT_CUDA(cudaStreamSynchronize(st));
    if (ptr) cudaFree(ptr);
    ptr = p;
    cap = want;
    return GTGPU_OK;
}

DevMem::~DevMem() {
    if (ptr) cudaFree(ptr);
}

static KeySlots key_slots(DevMem& hash, DevMem& soff, DevMem& first_byte, DevMem& first, DevMem& klen, DevMem& known) {
    return KeySlots{(unsigned long long*)hash.ptr, (unsigned long long*)soff.ptr, (unsigned long long*)first_byte.ptr,
                    first.u32(), klen.u32(), known.u32()};
}

int32_t KeyTable::add_window(gtgpu_ctx* ctx, const char* d_text, uint64_t byte0, const ParsedLines& pl, uint32_t n_names) {
    const uint32_t nw = pl.n;
    if (nw == 0) return GTGPU_OK;
    cudaStream_t st = ctx->stream;
    const uint32_t base = (uint32_t)n;
    const size_t need = (size_t)(n + nw) * 4, have = (size_t)n * 4;
    for (DevMem* m : {&chr, &start, &end, &id}) GT_TRY(m->reserve(need, have, st));
    GT_CUDA(cudaMemcpyAsync(chr.u32() + base, pl.chr, (size_t)nw * 4, cudaMemcpyDeviceToDevice, st));
    GT_CUDA(cudaMemcpyAsync(start.u32() + base, pl.start, (size_t)nw * 4, cudaMemcpyDeviceToDevice, st));
    GT_CUDA(cudaMemcpyAsync(end.u32() + base, pl.end, (size_t)nw * 4, cudaMemcpyDeviceToDevice, st));
    // the table holds at most min(distinct + nw, max_keys) keys after this window (more are an error): keep it at most half full
    uint64_t new_cap = std::max<uint64_t>(cap, 1024);
    while (new_cap < 2 * std::min<uint64_t>(distinct + nw, max_keys)) new_cap <<= 1;
    if (new_cap != cap) {
        DevMem t_hash, t_soff, t_first_byte, t_first, t_klen, t_known;
        GT_TRY(t_hash.reserve(new_cap * 8, 0, st));
        GT_TRY(t_soff.reserve(new_cap * 8, 0, st));
        GT_TRY(t_first.reserve(new_cap * 4, 0, st));
        GT_TRY(t_klen.reserve(new_cap * 4, 0, st));
        if (record_spans) GT_TRY(t_first_byte.reserve(new_cap * 8, 0, st));
        if (!keep_all) {
            GT_TRY(t_known.reserve(new_cap * 4, 0, st));
            GT_CUDA(cudaMemsetAsync(t_known.ptr, 0, new_cap * 4, st));
        }
        GT_CUDA(cudaMemsetAsync(t_hash.ptr, 0, new_cap * 8, st));
        GT_CUDA(cudaMemsetAsync(t_first.ptr, 0xFF, new_cap * 4, st));
        if (cap) {
            ingest_key_rehash_kernel<<<grid_for(ctx, cap), 256, 0, st>>>(cap, key_slots(hash, soff, first_byte, first, klen, known),
                                                                     (uint32_t)(new_cap - 1),
                                                                     key_slots(t_hash, t_soff, t_first_byte, t_first, t_klen, t_known));
            ctx->launches++;
        }
        GT_CUDA(cudaStreamSynchronize(st));
        hash.swap(t_hash);
        soff.swap(t_soff);
        first_byte.swap(t_first_byte);
        first.swap(t_first);
        klen.swap(t_klen);
        known.swap(t_known);
        cap = new_cap;
    }
    const uint32_t mask = (uint32_t)(cap - 1);
    uint32_t *slot_of = pl.free[0], *wpos = pl.free[1], *wlen = pl.free[2];
    ingest_key_insert_kernel<<<grid_for(ctx, nw), 256, 0, st>>>(nw, pl.h, mask, (unsigned long long*)hash.ptr, first.u32(), slot_of, base,
                                                             pl.flags + 3);
    ingest_key_heads_kernel<<<grid_for(ctx, nw), 256, 0, st>>>(nw, base, slot_of, first.u32(), pl.chr, pl.bl, n_names, mask, id.u32(),
                                                            klen.u32(), known.u32(), wlen, pl.flags + 2);
    ctx->launches += 2;
    GT_TRY(exclusive_scan<uint32_t>(ctx, wlen, wpos, nw, pl.tmp));
    uint32_t tail[4];  // last offset, last length, keys first seen here, table full
    GT_CUDA(cudaMemcpyAsync(&tail[0], wpos + nw - 1, 4, cudaMemcpyDeviceToHost, st));
    GT_CUDA(cudaMemcpyAsync(&tail[1], wlen + nw - 1, 4, cudaMemcpyDeviceToHost, st));
    GT_CUDA(cudaMemcpyAsync(&tail[2], pl.flags + 2, 8, cudaMemcpyDeviceToHost, st));
    GT_CUDA(cudaStreamSynchronize(st));
    if (tail[3] || distinct + tail[2] > max_keys)
        return fail(GTGPU_ERR_UNSUPPORTED, who + ": more than " + std::to_string(max_keys) + " distinct " + keys);
    const uint64_t bytes = (uint64_t)tail[0] + tail[1];
    GT_TRY(arena.reserve(used + bytes + 1, used, st));
    ingest_key_claim_kernel<<<grid_for(ctx, nw), 256, 0, st>>>(nw, base, d_text, slot_of, id.u32(), pl.bo, pl.bl, wpos, used,
                                                            (char*)arena.ptr, (unsigned long long*)soff.ptr, byte0,
                                                            (unsigned long long*)first_byte.ptr);
    ingest_key_check_kernel<<<grid_for(ctx, nw), 256, 0, st>>>(nw, base, d_text, slot_of, id.u32(), pl.bo, pl.bl, klen.u32(),
                                                            (const char*)arena.ptr, (const unsigned long long*)soff.ptr, pl.flags + 1);
    ctx->launches += 2;
    uint32_t collision = 0;
    GT_CUDA(cudaMemcpyAsync(&collision, pl.flags + 1, 4, cudaMemcpyDeviceToHost, st));
    GT_CUDA(cudaStreamSynchronize(st));  // the window's text may be overwritten after this
    if (collision) return fail(GTGPU_ERR_UNSUPPORTED, who + ": two " + keys + " share a 64-bit hash; use " + array_entry);
    used += bytes;
    distinct += tail[2];
    n += nw;
    return GTGPU_OK;
}

int32_t KeyTable::finish(gtgpu_ctx* ctx, uint32_t* n_kept, BufPtr* out_names, BufPtr* out_name_offsets, BufPtr* out_spans) {
    cudaStream_t st = ctx->stream;
    uint32_t kept = 0;
    uint64_t blob_bytes = 0;
    char* d_blob = nullptr;
    unsigned long long* d_noff = nullptr;
    uint32_t* d_spans = nullptr;
    if (n) {
        // the kept keys' first appearances, sorted: key i of that order gets id i
        uint32_t *k_a, *v_a, *k_b, *v_b, *d_cnt;
        void* d_tmp;
        GT_TRY(ctx->scratch_get(SC_ING_0, distinct * 4, (void**)&k_a));
        GT_TRY(ctx->scratch_get(SC_ING_1, distinct * 4, (void**)&v_a));
        GT_TRY(ctx->scratch_get(SC_ING_2, distinct * 4, (void**)&k_b));
        GT_TRY(ctx->scratch_get(SC_ING_3, distinct * 4, (void**)&v_b));
        GT_TRY(ctx->scratch_get(SC_MISC, 64, (void**)&d_cnt));
        GT_CUDA(cudaMemsetAsync(d_cnt, 0, 4, st));
        ingest_key_kept_kernel<<<grid_for(ctx, cap), 256, 0, st>>>(cap, (const unsigned long long*)hash.ptr, first.u32(), known.u32(), k_a,
                                                                v_a, d_cnt);
        ctx->launches++;
        GT_CUDA(cudaMemcpyAsync(&kept, d_cnt, 4, cudaMemcpyDeviceToHost, st));
        GT_CUDA(cudaStreamSynchronize(st));
        GT_TRY(ctx->scratch_get(SC_IN3_START, std::max(radix_sort_temp_bytes(kept), exclusive_scan_temp_bytes(kept, 8)), &d_tmp));
        if (kept) {
            int in_b = 0;
            GT_TRY(radix_sort_pairs(ctx, kept, k_a, v_a, k_b, v_b, bits_for_value(n - 1), d_tmp, &in_b));
            if (in_b) { std::swap(k_a, k_b); std::swap(v_a, v_b); }
            unsigned long long* d_len = nullptr;
            if (out_spans) {
                GT_TRY(ctx->scratch_get(SC_FILE_OFFS, (uint64_t)kept * 8 + 8, (void**)&d_spans));
            } else {
                GT_TRY(ctx->scratch_get(SC_ING_4, (uint64_t)kept * 8, (void**)&d_len));
                GT_TRY(ctx->scratch_get(SC_ING_7, ((uint64_t)kept + 1) * 8, (void**)&d_noff));
            }
            ingest_key_lengths_kernel<<<grid_for(ctx, kept), 256, 0, st>>>(kept, v_a, klen.u32(), (const unsigned long long*)first_byte.ptr,
                                                                        d_len, d_spans);
            ctx->launches++;
            if (!out_spans) {
                GT_TRY(exclusive_scan<unsigned long long>(ctx, d_len, d_noff, kept, d_tmp));
                unsigned long long t64[2];
                GT_CUDA(cudaMemcpyAsync(&t64[0], d_noff + kept - 1, 8, cudaMemcpyDeviceToHost, st));
                GT_CUDA(cudaMemcpyAsync(&t64[1], d_len + kept - 1, 8, cudaMemcpyDeviceToHost, st));
                GT_CUDA(cudaStreamSynchronize(st));
                blob_bytes = t64[0] + t64[1];
                GT_TRY(ctx->scratch_get(SC_ING_6, blob_bytes + 1, (void**)&d_blob));
                ingest_key_names_kernel<<<grid_for(ctx, kept), 256, 0, st>>>(kept, v_a, klen.u32(), (const unsigned long long*)soff.ptr,
                                                                          (const char*)arena.ptr, d_noff, d_blob);
                ctx->launches++;
            }
        }
        ingest_key_ids_kernel<<<grid_for(ctx, n), 256, 0, st>>>(n, k_a, kept, id.u32());
        ctx->launches++;
        GT_CUDA(cudaGetLastError());
    }
    *n_kept = kept;
    if (out_spans) {
        BufPtr spans;
        int32_t s = buf_from_device(ctx, d_spans, (uint64_t)kept * 2, 4, st, &spans);
        if (s == GTGPU_ERR_CUDA) return fail(s, who + ": D2H of the " + key + " spans failed");
        GT_TRY(s);
        if (cudaStreamSynchronize(st) != cudaSuccess) return fail(GTGPU_ERR_CUDA, who + ": D2H of the " + key + " spans failed");
        *out_spans = std::move(spans);
        return GTGPU_OK;
    }
    BufPtr names, offsets;
    int32_t s = buf_from_device(ctx, d_blob, blob_bytes, 1, st, &names);
    if (s == GTGPU_ERR_CUDA) return fail(s, who + ": D2H of the " + key + " names failed");
    GT_TRY(s);
    s = buf_new(ctx, (uint64_t)kept + 1, 8, &offsets);  // the last offset is written on the host
    if (s == GTGPU_OK && kept && cudaMemcpyAsync(offsets->block.ptr, d_noff, (uint64_t)kept * 8, cudaMemcpyDeviceToHost, st) != cudaSuccess)
        s = fail(GTGPU_ERR_CUDA, who + ": D2H of the " + key + " name offsets failed");
    if (s == GTGPU_OK && cudaStreamSynchronize(st) != cudaSuccess) s = fail(GTGPU_ERR_CUDA, who + ": D2H failed");
    if (s != GTGPU_OK) {
        cudaStreamSynchronize(st);  // the names' copy may still run
        return s;
    }
    reinterpret_cast<uint64_t*>(offsets->block.ptr)[kept] = blob_bytes;
    *out_names = std::move(names);
    *out_name_offsets = std::move(offsets);
    return GTGPU_OK;
}

// The fragment lines of tokenize_fragment_file (fragments.rs:12-56) from a fragment file's text of any size: every window is
// parsed and its fragments and barcodes go into *tab, a KeyTable that keeps every barcode.  The caller holds ctx->mu.
static int32_t parse_fragment_file_locked(gtgpu_ctx* ctx, const Text& t, uint32_t n_names, const char* names, const uint32_t* name_offsets,
                                          const std::string& who, KeyTable* tab) {
    if (t.n_bytes == 0) return GTGPU_OK;
    NameTable nt;
    GT_TRY(upload_name_table(ctx, n_names, names, name_offsets, &nt));
    return for_each_window(ctx, t, who, [&](const char* d, uint64_t nb, uint64_t byte0, uint64_t line0, uint32_t* n_lines) -> int32_t {
        ParsedLines fp;
        GT_TRY(parse_lines_locked(ctx, d, nb, FRAG_TOKENIZE, nt, BedFilesView{}, &fp));
        *n_lines = fp.n_lines;
        if (fp.bad_line != 0xFFFFFFFFu)
            return fail(GTGPU_ERR_INVALID, who + ": Invalid fragment file detected at line: " + std::to_string(line0 + fp.bad_line));
        if (tab->n + fp.n > 0xFFFFFFFFull) return fail(GTGPU_ERR_UNSUPPORTED, who + ": more than 2^32 - 1 fragments in one file");
        return tab->add_window(ctx, d, byte0, fp, n_names);
    });
}

// tokenize_fragment_file (fragments.rs:61-82) from a fragment file's text of any size: after the windowed parse the fragment
// tokenizer core runs once over the accumulated fragments and their dense barcode ids.  With out_spans the barcodes come back
// as u32 (first byte, length) spans into the text, else as names + u64 name offsets.  The caller holds ctx->mu.
static int32_t tokenize_fragments_file_locked(gtgpu_index* ix, const Text& t, uint32_t n_names, const char* names,
                                              const uint32_t* name_offsets, uint32_t unk_id, const std::string& who, uint32_t* out_n_barcodes,
                                              BufPtr* out_names, BufPtr* out_name_offsets, BufPtr* out_spans, BufPtr* out_barcode_offsets,
                                              BufPtr* out_ids) {
    gtgpu_ctx* ctx = ix->ctx;
    KeyTable tab(true, out_spans != nullptr, ~0ull, who, "gtgpu_tokenize_fragments", "barcode", "barcodes");
    GT_TRY(parse_fragment_file_locked(ctx, t, n_names, names, name_offsets, who, &tab));
    uint32_t n_barcodes = 0;
    BufPtr offs, ids;
    GT_TRY(tab.finish(ctx, &n_barcodes, out_names, out_name_offsets, out_spans));
    GT_TRY(buf_new(ctx, (uint64_t)n_barcodes + 1, 8, &offs));
    GT_TRY(tokenize_fragments_core(ix, tab.n, tab.chr.u32(), tab.start.u32(), tab.end.u32(), tab.id.u32(), n_barcodes, unk_id,
                                   (uint64_t*)offs->block.ptr, &ids));
    *out_n_barcodes = n_barcodes;
    *out_barcode_offsets = std::move(offs);
    *out_ids = std::move(ids);
    return GTGPU_OK;
}

// ---- the BED files of an IGD database: region lines of many files, chromosome names discovered on the device ------------------
// The names go through a KeyTable that keeps every name (an assembly names 25 to ~1e5 contigs; at most MAX_CHROM_NAMES).
constexpr uint64_t MAX_CHROM_NAMES = 1u << 18;

// records are in file order: file f's records start at the first record whose file is >= f
__global__ void ingest_file_record_offsets_kernel(uint64_t n_files, const uint32_t* __restrict__ file, uint64_t n,
                                                  unsigned long long* __restrict__ out) {
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t f = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; f <= n_files; f += stride) {
        uint64_t lo = 0, hi = n;
        while (lo < hi) {
            const uint64_t mid = (lo + hi) >> 1;
            if (file[mid] < f) lo = mid + 1;
            else hi = mid;
        }
        out[f] = lo;
    }
}

int32_t parse_bed_files_locked(gtgpu_ctx* ctx, const Text& t, const std::string& who, BedFilesRecords* out) {
    cudaStream_t st = ctx->stream;
    const uint64_t n_files = t.n_files, *file_offsets = t.file_offsets.data();
    DevMem d_fo, d_first_line, d_fs;
    GT_TRY(d_fo.reserve((n_files + 1) * 8, 0, st));
    GT_TRY(d_first_line.reserve(std::max<uint64_t>(n_files, 1) * 8, 0, st));
    GT_CUDA(cudaMemcpyAsync(d_fo.ptr, file_offsets, (n_files + 1) * 8, cudaMemcpyHostToDevice, st));
    GT_CUDA(cudaStreamSynchronize(st));  // file_offsets is the caller's
    KeyTable tab(true, false, MAX_CHROM_NAMES, who, "gtgpu_igd_build", "chromosome", "chromosome names");
    std::vector<uint32_t> fs;  // the window's file starts that are not its first byte (window-relative)
    GT_TRY(for_each_window(ctx, t, who, [&](const char* d, uint64_t nb, uint64_t byte0, uint64_t line0, uint32_t* n_lines) -> int32_t {
        fs.clear();
        for (const uint64_t* f = std::upper_bound(file_offsets, file_offsets + n_files + 1, byte0);
             f < file_offsets + n_files + 1 && *f < byte0 + nb; ++f)
            if (fs.empty() || fs.back() != *f - byte0) fs.push_back((uint32_t)(*f - byte0));
        if (!fs.empty()) {
            GT_TRY(d_fs.reserve(fs.size() * 4, 0, st));
            GT_CUDA(cudaMemcpyAsync(d_fs.ptr, fs.data(), fs.size() * 4, cudaMemcpyHostToDevice, st));
        }
        BedFilesView fv;
        fv.file_offsets = (const unsigned long long*)d_fo.ptr;
        fv.n_files = n_files;
        fv.byte0 = byte0;
        fv.line0 = line0;
        fv.first_line = (unsigned long long*)d_first_line.ptr;
        fv.fstart = d_fs.u32();
        fv.n_fstart = (uint32_t)fs.size();
        ParsedLines pl;
        GT_TRY(parse_lines_locked(ctx, d, nb, BED_FILE_LINES, NameTable{}, fv, &pl));
        *n_lines = pl.n_lines;
        if (pl.bad_line != 0xFFFFFFFFu) {  // the file of the first malformed line and the line's number in that file
            const uint32_t li = pl.bad_line;
            uint32_t a = 0;
            if (li) GT_CUDA(cudaMemcpy(&a, pl.breaks + li - 1, 4, cudaMemcpyDeviceToHost));
            const uint64_t pos = byte0 + (li ? a + 1ull : 0ull);
            const uint64_t f = (uint64_t)(std::upper_bound(file_offsets, file_offsets + n_files, pos) - file_offsets) - 1;
            unsigned long long fl = 0;
            GT_CUDA(cudaMemcpy(&fl, (unsigned long long*)d_first_line.ptr + f, 8, cudaMemcpyDeviceToHost));
            return fail(GTGPU_ERR_INVALID, who + ": file " + std::to_string(f) + ", line " + std::to_string(line0 + li - fl + 1) +
                                               ": cannot parse start / end position (RegionParseError)");
        }
        if (pl.n && tab.n + pl.n >= 0xFFFFFFFFull) return fail(GTGPU_ERR_UNSUPPORTED, who + ": 2^32 - 1 region lines or more");
        return tab.add_window(ctx, d, byte0, pl, 0);
    }));
    // the table's chr column holds every record's file
    BedFilesRecords& r = *out;
    r.n = tab.n;
    r.file.swap(tab.chr);
    r.start.swap(tab.start);
    r.end.swap(tab.end);
    // ---- every file has a region line; records per file ---------------------------------------------------------------------
    r.file_offsets.assign(n_files + 1, 0);
    if (n_files) {
        DevMem roff;
        GT_TRY(roff.reserve((n_files + 1) * 8, 0, st));
        if (r.n) {
            ingest_file_record_offsets_kernel<<<grid_for(ctx, n_files + 1), 256, 0, st>>>(n_files, r.file.u32(), r.n,
                                                                                      (unsigned long long*)roff.ptr);
            ctx->launches++;
            GT_CUDA(cudaMemcpyAsync(r.file_offsets.data(), roff.ptr, (n_files + 1) * 8, cudaMemcpyDeviceToHost, st));
            GT_CUDA(cudaStreamSynchronize(st));
        }
        for (uint64_t f = 0; f < n_files; ++f)
            if (r.file_offsets[f + 1] == r.file_offsets[f])
                return fail(GTGPU_ERR_INVALID, who + ": file " + std::to_string(f) + ": Corrupted file. 0 regions found");
    }
    // ---- chromosome ids in first-appearance order ----------------------------------------------------------------------------
    GT_TRY(tab.finish(ctx, &r.n_names, &r.names, &r.name_offsets));
    r.chr.swap(tab.id);
    return GTGPU_OK;
}

// ---- query BED files: the discovered names mapped to the caller's ids ---------------------------------------------------------
// parse_bed_files_locked numbers the files' chromosome names in their first appearance; one launch maps every such name to the
// caller's id (its name table, looked up as gtgpu_parse_bed does), one more rewrites every record's chr.
__global__ void ingest_map_names_kernel(uint32_t n_names, const char* __restrict__ blob, const unsigned long long* __restrict__ offs,
                                        NameTable nt, uint32_t* __restrict__ map) {
    const uint32_t stride = gridDim.x * blockDim.x;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n_names; i += stride) {
        const char* s = blob + offs[i];
        const uint32_t len = (uint32_t)(offs[i + 1] - offs[i]);
        map[i] = nt.lookup(fnv1a64(s, len), s, len);
    }
}

// out[i] = map[in[i]] (in may be out)
__global__ void ingest_remap_chr_kernel(uint64_t n, const uint32_t* __restrict__ map, const uint32_t* in, uint32_t* out) {
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) out[i] = map[in[i]];
}

// The r->n records' discovered name ids in_chr -> the caller's ids in out_chr (r->chr, or any other column of the records).
static int32_t map_query_names_locked(gtgpu_ctx* ctx, const BedFilesRecords* r, uint32_t n_names, const char* names,
                                      const uint32_t* name_offsets, bool with_rank, NameTable* nt, const uint32_t* in_chr,
                                      uint32_t* out_chr) {
    cudaStream_t st = ctx->stream;
    GT_TRY(upload_name_table(ctx, n_names, names, name_offsets, nt, with_rank));  // scratch SC_SET_ID
    const uint64_t blob_bytes = r->names->len;
    DevMem d_blob, d_offs, d_map;
    GT_TRY(d_blob.reserve(std::max<uint64_t>(blob_bytes, 1), 0, st));
    GT_TRY(d_offs.reserve(((uint64_t)r->n_names + 1) * 8, 0, st));
    GT_TRY(d_map.reserve((uint64_t)r->n_names * 4, 0, st));
    if (blob_bytes) GT_CUDA(cudaMemcpyAsync(d_blob.ptr, r->names->block.ptr, blob_bytes, cudaMemcpyHostToDevice, st));
    GT_CUDA(cudaMemcpyAsync(d_offs.ptr, r->name_offsets->block.ptr, ((uint64_t)r->n_names + 1) * 8, cudaMemcpyHostToDevice, st));
    ingest_map_names_kernel<<<grid_for(ctx, r->n_names), 256, 0, st>>>(r->n_names, (const char*)d_blob.ptr,
                                                                     (const unsigned long long*)d_offs.ptr, *nt, d_map.u32());
    ingest_remap_chr_kernel<<<grid_for(ctx, r->n), 256, 0, st>>>(r->n, d_map.u32(), in_chr, out_chr);
    ctx->launches += 2;
    GT_CUDA(cudaGetLastError());
    GT_CUDA(cudaStreamSynchronize(st));  // the map is freed here, and a later call may reuse the name table's scratch
    return GTGPU_OK;
}

int32_t parse_bed_queries_locked(gtgpu_ctx* ctx, const Text& t, uint32_t n_names, const char* names, const uint32_t* name_offsets,
                                 bool with_rank, const std::string& who, BedFilesRecords* r, NameTable* nt) {
    GT_TRY(parse_bed_files_locked(ctx, t, who, r));
    if (r->n == 0) return GTGPU_OK;
    return map_query_names_locked(ctx, r, n_names, names, name_offsets, with_rank, nt, r->chr.u32(), r->chr.u32());
}

// ---- a batch of BED files tokenized in one pass: parse, per-file RegionSet::sort, fused find, [unk] rule ----------------------
// gtgpu_tokenize_bed_files on t.n_files > 0 files: out_file_token_offsets (n_files + 1, host) and *out_ids as gtgpu_tokenize_files
// returns them.  The records arrive grouped by file in file order.  The caller holds ctx->mu.
static int32_t tokenize_bed_files_locked(gtgpu_index* ix, const Text& t, uint32_t n_names, const char* names, const uint32_t* name_offsets,
                                         uint32_t unk_id, const std::string& who, uint64_t* out_file_token_offsets, BufPtr* out_ids) {
    gtgpu_ctx* ctx = ix->ctx;
    cudaStream_t st = ctx->stream;
    const uint64_t n_files = t.n_files;
    BedFilesRecords r;
    NameTable nt{};
    GT_TRY(parse_bed_queries_locked(ctx, t, n_names, names, name_offsets, true, who, &r, &nt));
    const uint32_t n = (uint32_t)r.n;  // parse_bed_files_locked allows fewer than 2^32 - 1 records
    const uint32_t *q_chr = r.chr.u32(), *q_start = r.start.u32(), *q_end = r.end.u32();
    GT_TRY(sort_regions_locked(ctx, n, nt, n_names, r.file.u32(), n_files, &q_chr, &q_start, &q_end));
    // ---- fused find over the files, then the [unk] rule (Tokenizer::tokenize: a file without a token yields [unk]) ----------------
    uint64_t *d_fo, *d_raw_tok, *d_out_tok, total = 0;
    GT_TRY(ctx->scratch_get(SC_FILE_OFFS, (n_files + 1) * 8, (void**)&d_fo));
    GT_TRY(ctx->scratch_get(SC_FILE_TOK, (n_files + 1) * 8, (void**)&d_raw_tok));
    GT_TRY(ctx->scratch_get(SC_FILE_TOK2, (n_files + 1) * 8, (void**)&d_out_tok));
    GT_CUDA(cudaMemcpyAsync(d_fo, r.file_offsets.data(), (n_files + 1) * 8, cudaMemcpyHostToDevice, st));
    uint32_t *d_ids = nullptr, *d_ids2 = nullptr;
    GT_TRY(fused_find_all(ix, n, n_files, d_fo, q_chr, q_start, q_end, nullptr, d_raw_tok, &d_ids, &total));  // synchronises
    uint64_t* d_misc;
    GT_TRY(ctx->scratch_get(SC_MISC, 64, (void**)&d_misc));
    GT_TRY(ctx->scratch_get(SC_OUT_IDS2, (total + n_files) * 4 + 4, (void**)&d_ids2));
    GT_TRY(launch_unk_offsets(ctx, n_files, d_raw_tok, d_out_tok, d_misc + 1));
    GT_TRY(launch_unk_expand(ctx, n_files, d_raw_tok, d_out_tok, d_ids, unk_id, d_ids2));
    GT_CUDA(cudaMemcpyAsync(out_file_token_offsets, d_out_tok, (n_files + 1) * 8, cudaMemcpyDeviceToHost, st));
    GT_CUDA(cudaStreamSynchronize(st));
    BufPtr buf;
    int32_t s = buf_from_device(ctx, d_ids2, out_file_token_offsets[n_files], 4, st, &buf);
    if (s == GTGPU_ERR_CUDA) return fail(s, who + ": D2H: " + gtgpu_last_error());
    GT_TRY(s);
    const cudaError_t e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) return fail(GTGPU_ERR_CUDA, who + ": D2H: " + cudaGetErrorString(e));
    *out_ids = std::move(buf);
    return GTGPU_OK;
}

// the caller holds ctx->mu
static int32_t tokenize_bed_locked(gtgpu_index* ix, const Text& t, uint32_t n_names, const char* names, const uint32_t* name_offsets,
                                   uint32_t unk_id, gtgpu_buf** out_ids) {
    gtgpu_ctx* ctx = ix->ctx;
    const uint32_t *d_chr, *d_start, *d_end;
    uint32_t* d_ids = nullptr;
    uint64_t n = 0, total = 0;
    GT_TRY(parse_bed_locked(ctx, t, n_names, names, name_offsets, &n, &d_chr, &d_start, &d_end));
    GT_TRY(fused_find_all(ix, n, 0, nullptr, d_chr, d_start, d_end, nullptr, nullptr, &d_ids, &total));
    BufPtr buf;
    if (total == 0) {  // Tokenizer::tokenize: a call without a single token yields [unk] (tokenizer.rs:156-160)
        GT_TRY(buf_new(ctx, 1, 4, &buf));
        *reinterpret_cast<uint32_t*>(buf->block.ptr) = unk_id;
        *out_ids = buf.release();
        return GTGPU_OK;
    }
    const int32_t s = buf_from_device(ctx, d_ids, total, 4, ctx->stream, &buf);
    if (s == GTGPU_ERR_CUDA) return fail(s, std::string("ingest: D2H: ") + gtgpu_last_error());
    GT_TRY(s);
    const cudaError_t e = cudaStreamSynchronize(ctx->stream);
    if (e != cudaSuccess) return fail(GTGPU_ERR_CUDA, std::string("ingest: D2H: ") + cudaGetErrorString(e));
    *out_ids = buf.release();
    return GTGPU_OK;
}

// ---- a batch of BED files against an overlap index: count / any / find / subset per file -------------------------------------
// Per-query outputs make the query order visible, and RegionSet::try_from sorts by (chromosome STRING, start) over every name of
// the file, names the index lacks included (region_set.rs:502-505).  So the records are sorted while their chr column still
// holds the names discovered in the files, ranked here by their bytes, and only then mapped to the caller's ids.

// hit i of the fused find's per-file runs (file_hits: n_files + 1 raw offsets): its key (keys[val], or val) and its file.
// fold: one word file << key_bits | key for a single radix pass; otherwise the key, with the file as the pair's value.
__global__ void overlaps_subset_keys_kernel(uint64_t total, const uint32_t* __restrict__ ids, const uint32_t* __restrict__ keys,
                                            uint64_t n_files, const unsigned long long* __restrict__ file_hits, int key_bits, bool fold,
                                            uint32_t* __restrict__ k, uint32_t* __restrict__ v) {
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
        const uint32_t key = keys ? keys[ids[i]] : ids[i];
        uint64_t lo = 0, hi = n_files;  // the last file whose hits start at or before i (files without hits start where the next does)
        while (hi - lo > 1) {
            const uint64_t mid = (lo + hi) >> 1;
            if (file_hits[mid] <= i) lo = mid;
            else hi = mid;
        }
        const uint32_t f = (uint32_t)lo;
        k[i] = fold ? f << key_bits | key : key;
        v[i] = f;
    }
}

// 1 where a new (file, key) starts in the sorted hits (file == nullptr: key holds the folded words)
__global__ void overlaps_subset_heads_kernel(uint64_t n, const uint32_t* __restrict__ key, const uint32_t* __restrict__ file,
                                             uint32_t* __restrict__ head) {
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride)
        head[i] = i == 0 || key[i] != key[i - 1] || (file && file[i] != file[i - 1]);
}

// the distinct (file, key) pairs at their scanned positions: keys to out_key, files to out_file (for the per-file offsets)
__global__ void overlaps_subset_unique_kernel(uint64_t n, const uint32_t* __restrict__ key, const uint32_t* __restrict__ file,
                                              const uint32_t* __restrict__ head, const uint32_t* __restrict__ pos, int key_bits,
                                              uint32_t* __restrict__ out_key, uint32_t* __restrict__ out_file) {
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride)
        if (head[i]) {
            const uint32_t q = pos[i], w = key[i];
            out_key[q] = file ? w : w & ((1u << key_bits) - 1u);
            out_file[q] = file ? file[i] : w >> key_bits;
        }
}

// ranks of the discovered names in byte order (Rust's String order)
static std::vector<uint32_t> name_byte_ranks(const BedFilesRecords& r) {
    const char* blob = (const char*)r.names->block.ptr;
    const uint64_t* off = (const uint64_t*)r.name_offsets->block.ptr;
    std::vector<uint32_t> by_name(r.n_names), rank(r.n_names);
    std::iota(by_name.begin(), by_name.end(), 0u);
    auto name = [&](uint32_t i) { return std::string_view(blob + off[i], off[i + 1] - off[i]); };
    std::sort(by_name.begin(), by_name.end(), [&](uint32_t a, uint32_t b) { return name(a) < name(b); });  // names are distinct
    for (uint32_t k = 0; k < r.n_names; ++k) rank[by_name[k]] = k;
    return rank;
}

// SUBSET: the ascending distinct keys of every file's hits.  The total hits (which can exceed the queries many times) size the
// scratch; they are sorted by (file, key) in one radix pass when both fit 32 bits, else by key and then by file.
static int32_t subset_reduce_locked(gtgpu_index* ix, uint64_t n_files, const uint32_t* d_ids, uint64_t total, const uint64_t* d_file_hits,
                                    const uint32_t* d_keys, uint32_t max_key, const std::string& who, BufPtr* out_offsets,
                                    BufPtr* out_values) {
    gtgpu_ctx* ctx = ix->ctx;
    cudaStream_t st = ctx->stream;
    if (total >= 0xFFFFFFFFull) return fail(GTGPU_ERR_UNSUPPORTED, who + ": 2^32 - 1 hits or more in one subset call");
    uint64_t* d_offs;
    uint32_t *out_key = nullptr, n_distinct = 0;
    GT_TRY(ctx->scratch_get(SC_FILE_TOK2, (n_files + 1) * 8, (void**)&d_offs));
    if (total == 0) {
        GT_CUDA(cudaMemsetAsync(d_offs, 0, (n_files + 1) * 8, st));
    } else {
        const int key_bits = bits_for_value(max_key), file_bits = bits_for_value(n_files - 1);
        const bool fold = key_bits + file_bits <= 32;
        uint32_t *k_a, *v_a, *k_b, *v_b, *head, *pos, *out_file;
        void* d_tmp;
        const size_t b = (size_t)total * 4;
        GT_TRY(ctx->scratch_get(SC_ING_0, b, (void**)&k_a));
        GT_TRY(ctx->scratch_get(SC_ING_1, b, (void**)&v_a));
        GT_TRY(ctx->scratch_get(SC_ING_2, b, (void**)&k_b));
        GT_TRY(ctx->scratch_get(SC_ING_3, b, (void**)&v_b));
        GT_TRY(ctx->scratch_get(SC_ING_4, b, (void**)&head));
        GT_TRY(ctx->scratch_get(SC_ING_5, b, (void**)&pos));
        GT_TRY(ctx->scratch_get(SC_ING_6, b, (void**)&out_file));
        GT_TRY(ctx->scratch_get(SC_OUT_IDS2, b, (void**)&out_key));
        GT_TRY(ctx->scratch_get(SC_IN3_START, std::max(radix_sort_temp_bytes(total), exclusive_scan_temp_bytes(total, 4)), &d_tmp));
        overlaps_subset_keys_kernel<<<grid_for(ctx, total), 256, 0, st>>>(total, d_ids, d_keys, n_files,
                                                                        (const unsigned long long*)d_file_hits, key_bits, fold, k_a, v_a);
        ctx->launches++;
        int in_b = 0;
        GT_TRY(radix_sort_pairs(ctx, total, k_a, v_a, k_b, v_b, fold ? key_bits + file_bits : key_bits, d_tmp, &in_b));
        if (in_b) { std::swap(k_a, k_b); std::swap(v_a, v_b); }
        const uint32_t *s_key = k_a, *s_file = nullptr;
        if (!fold) {  // stable by file: the files are the keys of this pass
            GT_TRY(radix_sort_pairs(ctx, total, v_a, k_a, v_b, k_b, file_bits, d_tmp, &in_b));
            s_key = in_b ? k_b : k_a;
            s_file = in_b ? v_b : v_a;
        }
        overlaps_subset_heads_kernel<<<grid_for(ctx, total), 256, 0, st>>>(total, s_key, s_file, head);
        ctx->launches++;
        GT_TRY(exclusive_scan<uint32_t>(ctx, head, pos, total, d_tmp));
        overlaps_subset_unique_kernel<<<grid_for(ctx, total), 256, 0, st>>>(total, s_key, s_file, head, pos, key_bits, out_key, out_file);
        ctx->launches++;
        uint32_t tail[2];
        GT_CUDA(cudaMemcpyAsync(&tail[0], pos + total - 1, 4, cudaMemcpyDeviceToHost, st));
        GT_CUDA(cudaMemcpyAsync(&tail[1], head + total - 1, 4, cudaMemcpyDeviceToHost, st));
        GT_CUDA(cudaStreamSynchronize(st));
        n_distinct = tail[0] + tail[1];
        ingest_file_record_offsets_kernel<<<grid_for(ctx, n_files + 1), 256, 0, st>>>(n_files, out_file, n_distinct,
                                                                                   (unsigned long long*)d_offs);
        ctx->launches++;
        GT_CUDA(cudaGetLastError());
    }
    GT_TRY(buf_from_device(ctx, d_offs, n_files + 1, 8, st, out_offsets));
    const int32_t s = buf_from_device(ctx, out_key, n_distinct, 4, st, out_values);
    const cudaError_t e = cudaStreamSynchronize(st);
    GT_TRY(s);
    if (e != cudaSuccess) return fail(GTGPU_ERR_CUDA, who + ": D2H: " + cudaGetErrorString(e));
    return GTGPU_OK;
}

// gtgpu_overlaps_bed_files on t.n_files > 0 files.  The caller holds ctx->mu.
static int32_t overlaps_bed_files_locked(gtgpu_index* ix, const Text& t, int32_t mode, uint32_t n_names, const char* names,
                                         const uint32_t* name_offsets, int32_t min_overlap, uint64_t n_keys, const uint32_t* keys,
                                         const std::string& who, uint64_t* out_file_queries, BufPtr* out_offsets, BufPtr* out_values) {
    gtgpu_ctx* ctx = ix->ctx;
    cudaStream_t st = ctx->stream;
    const uint64_t n_files = t.n_files;
    BedFilesRecords r;
    GT_TRY(parse_bed_files_locked(ctx, t, who, &r));
    const uint32_t n = (uint32_t)r.n;  // parse_bed_files_locked allows fewer than 2^32 - 1 records
    // ---- per file, stable by (name bytes, start); then the names in the caller's ids (into r.chr) ------------------------------
    // The sorted start / end may lie in scratch SC_ING_2 / SC_ING_3 (sort_regions_locked), which nothing touches before the
    // count or the fused find has read them.
    const uint32_t *q_chr = r.chr.u32(), *q_start = r.start.u32(), *q_end = r.end.u32();
    {
        const std::vector<uint32_t> rank = name_byte_ranks(r);
        DevMem d_rank;
        GT_TRY(d_rank.reserve((size_t)r.n_names * 4, 0, st));
        GT_CUDA(cudaMemcpyAsync(d_rank.ptr, rank.data(), (size_t)r.n_names * 4, cudaMemcpyHostToDevice, st));
        NameTable by_bytes{};
        by_bytes.n_names = r.n_names;
        by_bytes.rank = d_rank.u32();
        GT_TRY(sort_regions_locked(ctx, n, by_bytes, r.n_names, r.file.u32(), n_files, &q_chr, &q_start, &q_end));
        GT_CUDA(cudaStreamSynchronize(st));  // the ranks are freed here
        NameTable nt{};
        GT_TRY(map_query_names_locked(ctx, &r, n_names, names, name_offsets, false, &nt, q_chr, r.chr.u32()));
        q_chr = r.chr.u32();
    }
    std::copy(r.file_offsets.begin(), r.file_offsets.end(), out_file_queries);
    const int32_t m = min_overlap > 1 ? min_overlap : 0;  // the reference filters only when min_overlap > 1
    if (mode == GTGPU_OVERLAPS_COUNT || mode == GTGPU_OVERLAPS_ANY) {
        const size_t elem = mode == GTGPU_OVERLAPS_COUNT ? 4 : 1;
        void* d_out;
        GT_TRY(ctx->scratch_get(SC_COUNTS, (size_t)n * elem, &d_out));
        GT_TRY(launch_count(ix, n, q_chr, q_start, q_end, m, mode == GTGPU_OVERLAPS_COUNT ? COUNT_U32 : COUNT_ANY_U8, d_out));
        const int32_t s = buf_from_device(ctx, d_out, n, (uint32_t)elem, st, out_values);
        const cudaError_t e = cudaStreamSynchronize(st);
        GT_TRY(s);
        if (e != cudaSuccess) return fail(GTGPU_ERR_CUDA, who + ": " + cudaGetErrorString(e));
        return GTGPU_OK;
    }
    uint32_t* d_ids = nullptr;
    uint64_t total = 0;
    if (mode == GTGPU_OVERLAPS_FIND) {
        uint64_t* d_offsets;
        GT_TRY(ctx->scratch_get(SC_OUT_OFFS, ((uint64_t)n + 1) * 8, (void**)&d_offsets));
        GT_TRY(fused_find_all(ix, n, 0, nullptr, q_chr, q_start, q_end, d_offsets, nullptr, &d_ids, &total, m));  // synchronises
        GT_TRY(buf_from_device(ctx, d_offsets, (uint64_t)n + 1, 8, st, out_offsets));
        const int32_t s = buf_from_device(ctx, d_ids, total, 4, st, out_values);
        const cudaError_t e = cudaStreamSynchronize(st);
        GT_TRY(s);
        if (e != cudaSuccess) return fail(GTGPU_ERR_CUDA, who + ": D2H: " + cudaGetErrorString(e));
        return GTGPU_OK;
    }
    // ---- SUBSET ----------------------------------------------------------------------------------------------------------------
    uint32_t max_key = ix->max_val;
    DevMem d_keys;
    if (keys) {
        max_key = n_keys ? *std::max_element(keys, keys + n_keys) : 0u;
        GT_TRY(d_keys.reserve(n_keys * 4, 0, st));
        GT_CUDA(cudaMemcpyAsync(d_keys.ptr, keys, n_keys * 4, cudaMemcpyHostToDevice, st));
    }
    uint64_t *d_fo, *d_file_hits;
    GT_TRY(ctx->scratch_get(SC_FILE_OFFS, (n_files + 1) * 8, (void**)&d_fo));
    GT_TRY(ctx->scratch_get(SC_FILE_TOK, (n_files + 1) * 8, (void**)&d_file_hits));
    GT_CUDA(cudaMemcpyAsync(d_fo, r.file_offsets.data(), (n_files + 1) * 8, cudaMemcpyHostToDevice, st));
    GT_TRY(fused_find_all(ix, n, n_files, d_fo, q_chr, q_start, q_end, nullptr, d_file_hits, &d_ids, &total, m));  // synchronises
    return subset_reduce_locked(ix, n_files, d_ids, total, d_file_hits, keys ? d_keys.u32() : nullptr, max_key, who, out_offsets,
                                out_values);
}

// ---- the entry points: each plain-text / gzip pair shares one body ------------------------------------------------------------
// A body checks its arguments, takes ctx->mu, opens the text (open_text_locked: gzip members are inflated whole into device
// memory) and parses it where it is.  `who` is the entry point's name without "gtgpu_".

static int32_t tokenize_bed_text(gtgpu_index* ix, const TextIn& in, const char* who, uint32_t n_names, const char* names,
                                 const uint32_t* name_offsets, uint32_t unk_id, gtgpu_buf** out_ids) {
    if (!ix || !out_ids || (n_names && (!names || !name_offsets))) return fail(GTGPU_ERR_INVALID, std::string(who) + ": null argument");
    GT_TRY(in.check(who));
    gtgpu_ctx* ctx = ix->ctx;
    std::lock_guard<std::mutex> lk(ctx->mu);
    GT_CUDA(cudaSetDevice(ctx->device));
    Text t;
    GT_TRY(open_text_locked(ctx, in, who, &t));
    return tokenize_bed_locked(ix, t, n_names, names, name_offsets, unk_id, out_ids);
}

static int32_t tokenize_bed_files_text(gtgpu_index* ix, const TextIn& in, const char* who, uint32_t n_names, const char* names,
                                       const uint32_t* name_offsets, uint32_t unk_id, uint64_t* out_file_token_offsets,
                                       gtgpu_buf** out_ids) {
    if (!ix || !out_file_token_offsets || !out_ids || (n_names && (!names || !name_offsets)))
        return fail(GTGPU_ERR_INVALID, std::string(who) + ": null argument");
    GT_TRY(in.check(who));
    gtgpu_ctx* ctx = ix->ctx;
    std::lock_guard<std::mutex> lk(ctx->mu);
    GT_CUDA(cudaSetDevice(ctx->device));
    BufPtr ids;
    if (in.n_files == 0) {  // the offsets are [0] and the id buffer is empty
        GT_TRY(buf_new(ctx, 0, 4, &ids));
        out_file_token_offsets[0] = 0;
    } else {
        Text t;
        GT_TRY(open_text_locked(ctx, in, who, &t));
        GT_TRY(tokenize_bed_files_locked(ix, t, n_names, names, name_offsets, unk_id, who, out_file_token_offsets, &ids));
    }
    *out_ids = ids.release();
    return GTGPU_OK;
}

static int32_t overlaps_bed_files_text(gtgpu_index* ix, const TextIn& in, const char* who, int32_t mode, uint32_t n_names,
                                       const char* names, const uint32_t* name_offsets, int32_t min_overlap, uint64_t n_keys,
                                       const uint32_t* keys, uint64_t* out_file_queries, gtgpu_buf** out_offsets, gtgpu_buf** out_values) {
    const bool per_query = mode == GTGPU_OVERLAPS_COUNT || mode == GTGPU_OVERLAPS_ANY;
    if (mode < GTGPU_OVERLAPS_COUNT || mode > GTGPU_OVERLAPS_SUBSET) return fail(GTGPU_ERR_INVALID, std::string(who) + ": unknown mode");
    if (!ix || !out_file_queries || !out_values || (!per_query && !out_offsets) || (n_names && (!names || !name_offsets)) ||
        (n_keys && !keys))
        return fail(GTGPU_ERR_INVALID, std::string(who) + ": null argument");
    if (mode == GTGPU_OVERLAPS_SUBSET && keys && n_keys <= ix->max_val)
        return fail(GTGPU_ERR_INVALID, std::string(who) + ": keys must have an entry for every val of the index (n_keys > " +
                                           std::to_string(ix->max_val) + ")");
    GT_TRY(in.check(who));
    gtgpu_ctx* ctx = ix->ctx;
    std::lock_guard<std::mutex> lk(ctx->mu);
    GT_CUDA(cudaSetDevice(ctx->device));
    BufPtr offsets, values;
    if (in.n_files == 0) {  // the offsets are [0] and the buffers empty
        out_file_queries[0] = 0;
        GT_TRY(buf_new(ctx, 0, mode == GTGPU_OVERLAPS_ANY ? 1 : 4, &values));
        if (!per_query) {
            GT_TRY(buf_new(ctx, 1, 8, &offsets));
            *reinterpret_cast<uint64_t*>(offsets->block.ptr) = 0;
        }
    } else {
        Text t;
        GT_TRY(open_text_locked(ctx, in, who, &t));
        GT_TRY(overlaps_bed_files_locked(ix, t, mode, n_names, names, name_offsets, min_overlap, n_keys,
                                         mode == GTGPU_OVERLAPS_SUBSET ? keys : nullptr, who, out_file_queries, &offsets, &values));
    }
    if (out_offsets) *out_offsets = offsets.release();
    *out_values = values.release();
    return GTGPU_OK;
}

// tokenize_fragment_file (fragments.rs:61-82) from the file's text, < 4 GiB: the barcodes come back as u32 spans into the text.
// With out_text (gzip input) the inflated text comes back too, its copy on copy_out overlapping the parse.  The parse's errors
// carry the text form's name.
static int32_t tokenize_fragments_spans(gtgpu_index* ix, const TextIn& in, const char* who, uint32_t n_names, const char* names,
                                        const uint32_t* name_offsets, uint32_t unk_id, uint32_t* out_n_barcodes,
                                        gtgpu_buf** out_barcode_spans, gtgpu_buf** out_barcode_offsets, gtgpu_buf** out_ids,
                                        gtgpu_buf** out_text) {
    if (!ix || !out_n_barcodes || !out_barcode_spans || !out_barcode_offsets || !out_ids || (in.is_gz && !out_text) ||
        (n_names && (!names || !name_offsets)))
        return fail(GTGPU_ERR_INVALID, std::string(who) + ": null argument");
    GT_TRY(in.check(who));
    gtgpu_ctx* ctx = ix->ctx;
    std::lock_guard<std::mutex> lk(ctx->mu);
    GT_CUDA(cudaSetDevice(ctx->device));
    Text t;
    GT_TRY(open_text_locked(ctx, in, who, &t));
    if (t.n_bytes >= 0xFFFFFFF0ull) return fail(GTGPU_ERR_UNSUPPORTED, "tokenize_fragments_text: at most 4 GiB of text per call");
    BufPtr text, spans, offs, ids;
    int32_t s = GTGPU_OK;
    if (out_text) {
        s = buf_from_device(ctx, t.bytes, t.n_bytes, 1, ctx->copy_out, &text);
        if (s == GTGPU_ERR_CUDA) return fail(s, std::string(who) + ": D2H of the text failed");
        GT_TRY(s);
    }
    try {
        s = tokenize_fragments_file_locked(ix, t, n_names, names, name_offsets, unk_id, "tokenize_fragments_text", out_n_barcodes, nullptr,
                                           nullptr, &spans, &offs, &ids);
    } catch (...) {
        cudaStreamSynchronize(ctx->copy_out);  // the text's copy ends before its block goes back to the cache
        throw;
    }
    if (s == GTGPU_OK && out_text && cudaStreamSynchronize(ctx->copy_out) != cudaSuccess)
        s = fail(GTGPU_ERR_CUDA, std::string(who) + ": D2H of the text failed");
    if (s != GTGPU_OK) {
        cudaStreamSynchronize(ctx->copy_out);
        return s;
    }
    *out_barcode_spans = spans.release();
    *out_barcode_offsets = offs.release();
    *out_ids = ids.release();
    if (out_text) *out_text = text.release();
    return GTGPU_OK;
}

// tokenize_fragment_file from the file's text, any size: the barcodes come back as names.
static int32_t tokenize_fragments_names(gtgpu_index* ix, const TextIn& in, const char* who, uint32_t n_names, const char* names,
                                        const uint32_t* name_offsets, uint32_t unk_id, uint32_t* out_n_barcodes,
                                        gtgpu_buf** out_barcode_names, gtgpu_buf** out_barcode_name_offsets,
                                        gtgpu_buf** out_barcode_offsets, gtgpu_buf** out_ids) {
    if (!ix || !out_n_barcodes || !out_barcode_names || !out_barcode_name_offsets || !out_barcode_offsets || !out_ids ||
        (n_names && (!names || !name_offsets)))
        return fail(GTGPU_ERR_INVALID, std::string(who) + ": null argument");
    GT_TRY(in.check(who));
    gtgpu_ctx* ctx = ix->ctx;
    std::lock_guard<std::mutex> lk(ctx->mu);
    GT_CUDA(cudaSetDevice(ctx->device));
    Text t;
    GT_TRY(open_text_locked(ctx, in, who, &t));
    BufPtr nm, no, offs, ids;
    GT_TRY(tokenize_fragments_file_locked(ix, t, n_names, names, name_offsets, unk_id, who, out_n_barcodes, &nm, &no, nullptr, &offs,
                                          &ids));
    *out_barcode_names = nm.release();
    *out_barcode_name_offsets = no.release();
    *out_barcode_offsets = offs.release();
    *out_ids = ids.release();
    return GTGPU_OK;
}

// count_fragments_by_barcode (fragments.rs:87-112) from the file's text, any size: the parse of tokenize_fragments_names, then
// per barcode its distinct token ids and their counts.
static int32_t count_fragments_file(gtgpu_index* ix, const TextIn& in, const char* who, uint32_t n_names, const char* names,
                                    const uint32_t* name_offsets, uint32_t unk_id, uint32_t* out_n_barcodes,
                                    gtgpu_buf** out_barcode_names, gtgpu_buf** out_barcode_name_offsets,
                                    gtgpu_buf** out_barcode_offsets, gtgpu_buf** out_tokens, gtgpu_buf** out_counts) {
    if (!ix || !out_n_barcodes || !out_barcode_names || !out_barcode_name_offsets || !out_barcode_offsets || !out_tokens || !out_counts ||
        (n_names && (!names || !name_offsets)))
        return fail(GTGPU_ERR_INVALID, std::string(who) + ": null argument");
    GT_TRY(in.check(who));
    gtgpu_ctx* ctx = ix->ctx;
    std::lock_guard<std::mutex> lk(ctx->mu);
    GT_CUDA(cudaSetDevice(ctx->device));
    Text t;
    GT_TRY(open_text_locked(ctx, in, who, &t));
    KeyTable tab(true, false, ~0ull, who, "gtgpu_tokenize_fragments", "barcode", "barcodes");
    GT_TRY(parse_fragment_file_locked(ctx, t, n_names, names, name_offsets, who, &tab));
    uint32_t n_barcodes = 0;
    BufPtr nm, no, offs;
    GT_TRY(tab.finish(ctx, &n_barcodes, &nm, &no));
    GT_TRY(buf_new(ctx, (uint64_t)n_barcodes + 1, 8, &offs));
    GT_TRY(count_fragments_core(ix, tab.n, tab.chr.u32(), tab.start.u32(), tab.end.u32(), tab.id.u32(), n_barcodes, unk_id,
                                (uint64_t*)offs->block.ptr, out_tokens, out_counts));
    *out_n_barcodes = n_barcodes;
    *out_barcode_names = nm.release();
    *out_barcode_name_offsets = no.release();
    *out_barcode_offsets = offs.release();
    return GTGPU_OK;
}

}  // namespace gtgpu

using namespace gtgpu;

extern "C" int32_t gtgpu_parse_bed(gtgpu_ctx* ctx, const char* text, uint64_t n_bytes, uint32_t n_names, const char* names,
                                   const uint32_t* name_offsets, uint64_t* out_n, gtgpu_buf** out_chr, gtgpu_buf** out_start,
                                   gtgpu_buf** out_end) try {
    if (!ctx || !out_n || !out_chr || !out_start || !out_end || (n_bytes && !text) || (n_names && (!names || !name_offsets)))
        return fail(GTGPU_ERR_INVALID, "parse_bed: null argument");
    std::lock_guard<std::mutex> lk(ctx->mu);
    GT_CUDA(cudaSetDevice(ctx->device));
    Text t;
    GT_TRY(open_text_locked(ctx, TextIn::plain(text, n_bytes), "parse_bed", &t));
    const uint32_t *d_chr, *d_start, *d_end;
    uint64_t n = 0;
    GT_TRY(parse_bed_locked(ctx, t, n_names, names, name_offsets, &n, &d_chr, &d_start, &d_end));
    BufPtr bufs[3];
    const uint32_t* src[3] = {d_chr, d_start, d_end};
    for (int k = 0; k < 3; ++k) {
        const int32_t s = buf_from_device(ctx, src[k], n, 4, ctx->stream, &bufs[k]);
        if (s == GTGPU_ERR_CUDA) return fail(s, std::string("ingest: D2H: ") + gtgpu_last_error());
        GT_TRY(s);
        const cudaError_t e = cudaStreamSynchronize(ctx->stream);
        if (e != cudaSuccess) return fail(GTGPU_ERR_CUDA, std::string("ingest: D2H: ") + cudaGetErrorString(e));
    }
    *out_n = n;
    *out_chr = bufs[0].release();
    *out_start = bufs[1].release();
    *out_end = bufs[2].release();
    return GTGPU_OK;
} GT_CATCH

extern "C" int32_t gtgpu_tokenize_bed(gtgpu_index* ix, const char* text, uint64_t n_bytes, uint32_t n_names, const char* names,
                                      const uint32_t* name_offsets, uint32_t unk_id, gtgpu_buf** out_ids) try {
    return tokenize_bed_text(ix, TextIn::plain(text, n_bytes), "tokenize_bed", n_names, names, name_offsets, unk_id, out_ids);
} GT_CATCH

// gtgpu_tokenize_bed on gzip members: inflate on the device, parse + sort + tokenize the text where it is.
extern "C" int32_t gtgpu_tokenize_bed_gz(gtgpu_index* ix, uint64_t n_members, const uint8_t* gz, const uint64_t* member_offsets,
                                         uint32_t n_names, const char* names, const uint32_t* name_offsets, uint32_t unk_id,
                                         gtgpu_buf** out_ids) try {
    return tokenize_bed_text(ix, TextIn::gzip(n_members, gz, member_offsets), "tokenize_bed_gz", n_names, names, name_offsets, unk_id,
                             out_ids);
} GT_CATCH

extern "C" int32_t gtgpu_tokenize_bed_files(gtgpu_index* ix, uint64_t n_files, const char* text, const uint64_t* file_offsets,
                                            uint32_t n_names, const char* names, const uint32_t* name_offsets, uint32_t unk_id,
                                            uint64_t* out_file_token_offsets, gtgpu_buf** out_ids) try {
    return tokenize_bed_files_text(ix, TextIn::plain(text, n_files, file_offsets), "tokenize_bed_files", n_names, names, name_offsets,
                                   unk_id, out_file_token_offsets, out_ids);
} GT_CATCH

extern "C" int32_t gtgpu_tokenize_bed_files_gz(gtgpu_index* ix, uint64_t n_files, const uint64_t* file_members, uint64_t n_members,
                                               const uint8_t* gz, const uint64_t* member_offsets, uint32_t n_names, const char* names,
                                               const uint32_t* name_offsets, uint32_t unk_id, uint64_t* out_file_token_offsets,
                                               gtgpu_buf** out_ids) try {
    return tokenize_bed_files_text(ix, TextIn::gzip(n_members, gz, member_offsets, n_files, file_members), "tokenize_bed_files_gz",
                                   n_names, names, name_offsets, unk_id, out_file_token_offsets, out_ids);
} GT_CATCH

extern "C" int32_t gtgpu_overlaps_bed_files(gtgpu_index* ix, int32_t mode, uint64_t n_files, const char* text, const uint64_t* file_offsets,
                                            uint32_t n_names, const char* names, const uint32_t* name_offsets, int32_t min_overlap,
                                            uint64_t n_keys, const uint32_t* keys, uint64_t* out_file_queries, gtgpu_buf** out_offsets,
                                            gtgpu_buf** out_values) try {
    return overlaps_bed_files_text(ix, TextIn::plain(text, n_files, file_offsets), "overlaps_bed_files", mode, n_names, names, name_offsets,
                                   min_overlap, n_keys, keys, out_file_queries, out_offsets, out_values);
} GT_CATCH

extern "C" int32_t gtgpu_overlaps_bed_files_gz(gtgpu_index* ix, int32_t mode, uint64_t n_files, const uint64_t* file_members,
                                               uint64_t n_members, const uint8_t* gz, const uint64_t* member_offsets, uint32_t n_names,
                                               const char* names, const uint32_t* name_offsets, int32_t min_overlap, uint64_t n_keys,
                                               const uint32_t* keys, uint64_t* out_file_queries, gtgpu_buf** out_offsets,
                                               gtgpu_buf** out_values) try {
    return overlaps_bed_files_text(ix, TextIn::gzip(n_members, gz, member_offsets, n_files, file_members), "overlaps_bed_files_gz", mode,
                                   n_names, names, name_offsets, min_overlap, n_keys, keys, out_file_queries, out_offsets, out_values);
} GT_CATCH

extern "C" int32_t gtgpu_tokenize_fragments_text(gtgpu_index* ix, const char* text, uint64_t n_bytes, uint32_t n_names,
                                                 const char* names, const uint32_t* name_offsets, uint32_t unk_id,
                                                 uint32_t* out_n_barcodes, gtgpu_buf** out_barcode_spans,
                                                 gtgpu_buf** out_barcode_offsets, gtgpu_buf** out_ids) try {
    return tokenize_fragments_spans(ix, TextIn::plain(text, n_bytes), "tokenize_fragments_text", n_names, names, name_offsets, unk_id,
                                    out_n_barcodes, out_barcode_spans, out_barcode_offsets, out_ids, nullptr);
} GT_CATCH

// gtgpu_tokenize_fragments_text on gzip members (a bgzip'ed fragment file: thousands of members).  *out_text returns the
// inflated text as well: the barcode spans index into it.
extern "C" int32_t gtgpu_tokenize_fragments_gz(gtgpu_index* ix, uint64_t n_members, const uint8_t* gz, const uint64_t* member_offsets,
                                               uint32_t n_names, const char* names, const uint32_t* name_offsets, uint32_t unk_id,
                                               uint32_t* out_n_barcodes, gtgpu_buf** out_barcode_spans,
                                               gtgpu_buf** out_barcode_offsets, gtgpu_buf** out_ids, gtgpu_buf** out_text) try {
    return tokenize_fragments_spans(ix, TextIn::gzip(n_members, gz, member_offsets), "tokenize_fragments_gz", n_names, names,
                                    name_offsets, unk_id, out_n_barcodes, out_barcode_spans, out_barcode_offsets, out_ids, out_text);
} GT_CATCH

extern "C" int32_t gtgpu_tokenize_fragments_file(gtgpu_index* ix, const char* text, uint64_t n_bytes, uint32_t n_names,
                                                 const char* names, const uint32_t* name_offsets, uint32_t unk_id,
                                                 uint32_t* out_n_barcodes, gtgpu_buf** out_barcode_names,
                                                 gtgpu_buf** out_barcode_name_offsets, gtgpu_buf** out_barcode_offsets,
                                                 gtgpu_buf** out_ids) try {
    return tokenize_fragments_names(ix, TextIn::plain(text, n_bytes), "tokenize_fragments_file", n_names, names, name_offsets, unk_id,
                                    out_n_barcodes, out_barcode_names, out_barcode_name_offsets, out_barcode_offsets, out_ids);
} GT_CATCH

extern "C" int32_t gtgpu_tokenize_fragments_file_gz(gtgpu_index* ix, uint64_t n_members, const uint8_t* gz, const uint64_t* member_offsets,
                                                    uint32_t n_names, const char* names, const uint32_t* name_offsets, uint32_t unk_id,
                                                    uint32_t* out_n_barcodes, gtgpu_buf** out_barcode_names,
                                                    gtgpu_buf** out_barcode_name_offsets, gtgpu_buf** out_barcode_offsets,
                                                    gtgpu_buf** out_ids) try {
    return tokenize_fragments_names(ix, TextIn::gzip(n_members, gz, member_offsets), "tokenize_fragments_file_gz", n_names, names,
                                    name_offsets, unk_id, out_n_barcodes, out_barcode_names, out_barcode_name_offsets,
                                    out_barcode_offsets, out_ids);
} GT_CATCH

extern "C" int32_t gtgpu_count_fragments_file(gtgpu_index* ix, const char* text, uint64_t n_bytes, uint32_t n_names, const char* names,
                                              const uint32_t* name_offsets, uint32_t unk_id, uint32_t* out_n_barcodes,
                                              gtgpu_buf** out_barcode_names, gtgpu_buf** out_barcode_name_offsets,
                                              gtgpu_buf** out_barcode_offsets, gtgpu_buf** out_tokens, gtgpu_buf** out_counts) try {
    return count_fragments_file(ix, TextIn::plain(text, n_bytes), "count_fragments_file", n_names, names, name_offsets, unk_id,
                                out_n_barcodes, out_barcode_names, out_barcode_name_offsets, out_barcode_offsets, out_tokens, out_counts);
} GT_CATCH

extern "C" int32_t gtgpu_count_fragments_file_gz(gtgpu_index* ix, uint64_t n_members, const uint8_t* gz, const uint64_t* member_offsets,
                                                 uint32_t n_names, const char* names, const uint32_t* name_offsets, uint32_t unk_id,
                                                 uint32_t* out_n_barcodes, gtgpu_buf** out_barcode_names,
                                                 gtgpu_buf** out_barcode_name_offsets, gtgpu_buf** out_barcode_offsets,
                                                 gtgpu_buf** out_tokens, gtgpu_buf** out_counts) try {
    return count_fragments_file(ix, TextIn::gzip(n_members, gz, member_offsets), "count_fragments_file_gz", n_names, names, name_offsets,
                                unk_id, out_n_barcodes, out_barcode_names, out_barcode_name_offsets, out_barcode_offsets, out_tokens,
                                out_counts);
} GT_CATCH
