// inflate.cu — gzip (RFC 1952 / DEFLATE RFC 1951) decoding on the device: gtgpu_gunzip.
//
// The reference reads `.gz` inputs through flate2's MultiGzDecoder (gtars-core/src/utils.rs:115-126): the text of a file is
// the concatenation of its gzip members.  A DEFLATE stream is sequential, so the parallelism here is ACROSS members: one
// warp inflates one member, thousands of members are in flight at once.  That is exactly the shape of the inputs on this
// path — a bgzip'ed fragment file is a chain of independent <= 64 KiB BGZF members (the BSIZE field of each header says
// where the next one starts, the ISIZE trailer how much text it holds), and a tokenization batch is thousands of small
// `.bed.gz` files of one member each — while a single multi-gigabyte one-member stream is not (the host layer keeps zlib
// for that).  With the text produced on the device, the ingest kernels (ingest.cu) parse it without it ever crossing PCIe.
//
// One warp per member, all 32 lanes run the Huffman decoder REDUNDANTLY (same bits, same control flow: no divergence, no
// broadcasts; table reads are shared-memory broadcasts), and split the byte work: input prefetch (512-byte segments, loaded
// into registers one segment ahead, committed to a 1 KiB shared-memory ring), literal runs and LZ77 copies.  The output
// window lives in global memory (a member's earlier text is read back through the L2 with ld.global.cg).
// Decoding tables per warp: a 10-bit first-level table for literal/length codes, a 9-bit one for distances, canonical
// count / symbol arrays for longer codes.  Every member's CRC-32 and ISIZE are verified (a corrupt member is an error, as
// in the reference).
#include <algorithm>
#include <cstring>
#include <vector>

#include "common.cuh"

namespace gtgpu {

namespace {

constexpr int INF_WARPS = 4;           // warps (= members) per block
constexpr int LL_BITS = 10, D_BITS = 9;
constexpr int RING = 1024, SEG = 512;  // input ring and prefetch segment (bytes)

struct WarpMem {
    uint8_t ring[RING];
    uint16_t ll_fast[1 << LL_BITS];  // sym | len << 9 (len 1..10), 0 = longer code
    uint16_t d_fast[1 << D_BITS];    // sym | len << 9
    uint16_t ll_sym[288], d_sym[32]; // symbols ordered by (code length, symbol)
    uint16_t ll_cnt[16], d_cnt[16];  // codes per length
    uint8_t len[320];                // code lengths while a dynamic header is read
    uint8_t lit[64];                 // pending literal run
};

__constant__ uint16_t c_len_base[29] = {3, 4, 5, 6, 7, 8, 9, 10, 11, 13, 15, 17, 19, 23, 27, 31, 35, 43, 51, 59, 67, 83, 99, 115, 131, 163, 195, 227, 258};
__constant__ uint8_t c_len_extra[29] = {0, 0, 0, 0, 0, 0, 0, 0, 1, 1, 1, 1, 2, 2, 2, 2, 3, 3, 3, 3, 4, 4, 4, 4, 5, 5, 5, 5, 0};
__constant__ uint16_t c_dist_base[30] = {1, 2, 3, 4, 5, 7, 9, 13, 17, 25, 33, 49, 65, 97, 129, 193, 257, 385, 513, 769, 1025, 1537, 2049, 3073, 4097, 6145, 8193, 12289, 16385, 24577};
__constant__ uint8_t c_dist_extra[30] = {0, 0, 0, 0, 1, 1, 2, 2, 3, 3, 4, 4, 5, 5, 6, 6, 7, 7, 8, 8, 9, 9, 10, 10, 11, 11, 12, 12, 13, 13};
__constant__ uint8_t c_clen_order[19] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};
__constant__ uint32_t c_crc_table[256];
__constant__ uint32_t c_crc_pow[32];  // x^(8 * 2^k) mod P, reflected: shifting a CRC over 2^k zero bytes

enum : uint32_t {
    INF_OK = 0, INF_BAD_HEADER = 1, INF_BAD_BLOCK = 2, INF_BAD_CODE = 3, INF_INPUT_END = 4, INF_OUTPUT_OVERRUN = 5,
    INF_BAD_DISTANCE = 6, INF_SIZE_MISMATCH = 7, INF_CRC_MISMATCH = 8, INF_TRAILING = 9,
};

// Reader state, identical in every lane of the warp.
struct Bits {
    uint64_t buf = 0;
    uint32_t cnt = 0;
    uint64_t pos = 0;       // next input byte (absolute offset into gz)
    uint64_t next_seg = 0;  // first byte that is not in the ring yet (its segment waits in `pre`)
    uint64_t end = 0;       // one past the member's last byte
    uint4 pre;              // this lane's 16 bytes of the prefetched segment
};

__device__ __forceinline__ uint4 load_seg(const uint8_t* gz, uint64_t seg, uint32_t lane) {
    return __ldg(reinterpret_cast<const uint4*>(gz + seg) + lane);  // gz is 512-byte aligned and padded past its end
}
__device__ __forceinline__ void store_seg(WarpMem& m, uint64_t seg, uint32_t lane, uint4 v) {
    *reinterpret_cast<uint4*>(m.ring + (seg & (RING - 1)) + lane * 16) = v;
}

__device__ __forceinline__ void ring_init(WarpMem& m, Bits& b, const uint8_t* gz, uint64_t pos, uint32_t lane) {
    __syncwarp();
    const uint64_t s0 = pos & ~(uint64_t)(SEG - 1);
    store_seg(m, s0, lane, load_seg(gz, s0, lane));
    store_seg(m, s0 + SEG, lane, load_seg(gz, s0 + SEG, lane));
    b.next_seg = s0 + 2 * SEG;
    b.pre = load_seg(gz, b.next_seg, lane);
    b.pos = pos;
    b.buf = 0;
    b.cnt = 0;
    __syncwarp();
}

// Keeps at least 32 bits in the buffer (a literal/length symbol with its extra bits needs 15 + 5, a distance 15 + 13).
__device__ __forceinline__ void refill(WarpMem& m, Bits& b, const uint8_t* gz, uint32_t lane) {
    if (b.cnt > 32) return;
    if (b.pos >= b.next_seg - SEG) {
        // the older half of the ring is consumed: commit the prefetched segment over it, request the one after
        __syncwarp();
        store_seg(m, b.next_seg, lane, b.pre);
        b.next_seg += SEG;
        b.pre = load_seg(gz, b.next_seg, lane);
        __syncwarp();
    }
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        b.buf |= (uint64_t)m.ring[(b.pos + k) & (RING - 1)] << (b.cnt + 8 * k);
    }
    b.pos += 4;
    b.cnt += 32;
}
__device__ __forceinline__ uint32_t peek(const Bits& b, uint32_t n) { return (uint32_t)b.buf & ((1u << n) - 1); }
__device__ __forceinline__ void drop(Bits& b, uint32_t n) {
    b.buf >>= n;
    b.cnt -= n;
}
__device__ __forceinline__ uint32_t take(WarpMem& m, Bits& b, const uint8_t* gz, uint32_t lane, uint32_t n) {
    refill(m, b, gz, lane);
    const uint32_t v = peek(b, n);
    drop(b, n);
    return v;
}
// bytes really consumed from the stream: whole bytes still in the bit buffer are given back
__device__ __forceinline__ uint64_t consumed(const Bits& b) { return b.pos - (b.cnt >> 3); }

__device__ __forceinline__ uint32_t bit_reverse(uint32_t v, uint32_t n) { return __brev(v) >> (32 - n); }

// Canonical Huffman tables from code lengths (RFC 1951 3.2.2): per-length counts, symbols ordered by (length, symbol) for
// the bit-by-bit path, and the first-level table for codes of at most FB bits.  Returns false for an over-subscribed set.
template <int FB>
__device__ bool build_tables(const uint8_t* len, uint32_t n, uint16_t* cnt, uint16_t* sym, uint16_t* fast, uint32_t lane) {
    __syncwarp();
    for (uint32_t i = lane; i < (1u << FB); i += 32) fast[i] = 0;
    __shared__ uint16_t s_offs_all[INF_WARPS][16];
    __shared__ uint16_t s_code_all[INF_WARPS][16];
    uint16_t* offs = s_offs_all[threadIdx.x >> 5];
    uint16_t* first_code = s_code_all[threadIdx.x >> 5];
    bool ok = true;
    if (lane == 0) {
        for (int l = 0; l < 16; ++l) cnt[l] = 0;
        for (uint32_t s = 0; s < n; ++s) cnt[len[s]]++;
        cnt[0] = 0;
        int left = 1;
        uint32_t code = 0, o = 0;
        for (int l = 1; l < 16; ++l) {
            left = (left << 1) - cnt[l];
            if (left < 0) ok = false;
            code = (code + cnt[l - 1]) << 1;
            first_code[l] = (uint16_t)code;
            offs[l] = (uint16_t)o;
            o += cnt[l];
        }
        if (ok)
            for (uint32_t s = 0; s < n; ++s)
                if (len[s]) sym[offs[len[s]]++] = (uint16_t)s;
        // offs[l] now = one past the last symbol of length l: restore the start
        if (ok)
            for (int l = 15, e = o; l >= 1; --l) {
                const int c = cnt[l];
                offs[l] = (uint16_t)(e - c);
                e -= c;
            }
    }
    ok = __shfl_sync(0xFFFFFFFFu, ok ? 1 : 0, 0) != 0;
    __syncwarp();
    if (!ok) return false;
    // first-level table: the k-th symbol (in symbol order) of length l has code first_code[l] + k
    for (int l = 1; l <= FB; ++l) {
        const uint32_t c = cnt[l], o = offs[l], fc = first_code[l];
        for (uint32_t k = lane; k < c; k += 32) {
            const uint32_t rev = bit_reverse(fc + k, l);
            const uint16_t e = (uint16_t)(sym[o + k] | (l << 9));
            for (uint32_t j = rev; j < (1u << FB); j += 1u << l) fast[j] = e;
        }
    }
    __syncwarp();
    return true;
}

// One symbol: first-level table, or the canonical bit-by-bit walk for codes longer than FB bits.  0xFFFF = invalid code.
template <int FB>
__device__ __forceinline__ uint32_t decode_sym(Bits& b, const uint16_t* fast, const uint16_t* cnt, const uint16_t* sym) {
    const uint32_t e = fast[peek(b, FB)];
    if (e) {
        drop(b, e >> 9);
        return e & 0x1FF;
    }
    int code = 0, first = 0, index = 0;  // signed on purpose: code - c < first must hold for code < c
    uint64_t bits = b.buf;
    for (uint32_t l = 1; l <= 15; ++l) {
        code |= (int)(bits & 1);
        bits >>= 1;
        const int c = cnt[l];
        if (code - c < first) {
            drop(b, l);
            return sym[index + (code - first)];
        }
        index += c;
        first += c;
        first <<= 1;
        code <<= 1;
    }
    return 0xFFFF;
}

__device__ __forceinline__ uint32_t crc_bytes(const uint32_t* table, const uint8_t* p, uint64_t n, uint32_t crc) {
    uint64_t i = 0;
    for (; i + 8 <= n; i += 8) {
        uint8_t v[8];
#pragma unroll
        for (int k = 0; k < 8; ++k) v[k] = __ldcg(p + i + k);  // eight loads in flight, then the dependent table chain
#pragma unroll
        for (int k = 0; k < 8; ++k) crc = table[(crc ^ v[k]) & 0xFF] ^ (crc >> 8);
    }
    for (; i < n; ++i) crc = table[(crc ^ __ldcg(p + i)) & 0xFF] ^ (crc >> 8);
    return crc;
}
// a(x) * b(x) mod P in the reflected representation zlib uses (crc32_combine's multmodp)
__device__ __forceinline__ uint32_t crc_mul(uint32_t a, uint32_t b) {
    uint32_t m = 1u << 31, p = 0;
    for (;;) {
        if (a & m) {
            p ^= b;
            if ((a & (m - 1)) == 0) break;
        }
        m >>= 1;
        b = (b & 1) ? (b >> 1) ^ 0xEDB88320u : b >> 1;
    }
    return p;
}
// CRC register after n further ZERO bytes
__device__ __forceinline__ uint32_t crc_shift(uint32_t crc, uint64_t n) {
    uint32_t p = 1u << 31;  // x^0
    for (int k = 0; n; ++k, n >>= 1)
        if (n & 1) p = crc_mul(c_crc_pow[k], p);
    return crc_mul(p, crc);
}

}  // namespace

// One warp per member.  status[k] = 0 or the INF_* code of the first problem in member k.
__global__ void __launch_bounds__(INF_WARPS * 32) gunzip_kernel(uint64_t n_members, const uint8_t* __restrict__ gz,
                                                                const uint64_t* __restrict__ member_offsets,
                                                                const uint64_t* __restrict__ out_offsets, uint8_t* out,
                                                                uint32_t* __restrict__ status) {
    __shared__ __align__(16) WarpMem s_mem[INF_WARPS];
    __shared__ uint32_t s_crc_table[256];  // per-lane slices index it with different bytes: shared memory, not constant
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    WarpMem& m = s_mem[warp];
    for (uint32_t i = threadIdx.x; i < 256; i += blockDim.x) s_crc_table[i] = c_crc_table[i];
    __syncthreads();
    for (uint64_t k = (uint64_t)blockIdx.x * INF_WARPS + warp; k < n_members; k += (uint64_t)gridDim.x * INF_WARPS) {
        const uint64_t in0 = member_offsets[k], in1 = member_offsets[k + 1];
        const uint64_t o0 = out_offsets[k], o1 = out_offsets[k + 1];
        uint32_t err = INF_OK;
        Bits b;
        b.end = in1;
        // ---- gzip header (RFC 1952 2.3): ID1 ID2 CM FLG MTIME(4) XFL OS [XLEN + extra] [name] [comment] [hcrc] ---------------
        uint64_t p = in0;
        if (in1 - in0 < 18 || gz[p] != 0x1F || gz[p + 1] != 0x8B || gz[p + 2] != 8 || (gz[p + 3] & 0xE0)) {
            err = INF_BAD_HEADER;
        } else {
            const uint32_t flg = gz[p + 3];
            p += 10;
            if (flg & 4) p += 2 + ((uint64_t)gz[p] | ((uint64_t)gz[p + 1] << 8));
            if (flg & 8) {
                while (p < in1 && gz[p]) ++p;
                ++p;
            }
            if (flg & 16) {
                while (p < in1 && gz[p]) ++p;
                ++p;
            }
            if (flg & 2) p += 2;
            if (p + 8 > in1) err = INF_BAD_HEADER;
        }
        uint64_t op = o0;  // next output byte
        uint32_t n_lit = 0;
        auto flush_lits = [&]() {
            if (n_lit) {
                for (uint32_t j = lane; j < n_lit; j += 32) out[op + j] = m.lit[j];
                op += n_lit;
                n_lit = 0;
                __syncwarp();
            }
        };
        if (!err) {
            ring_init(m, b, gz, p, lane);
            // ---- DEFLATE blocks ---------------------------------------------------------------------------------------------------
            for (bool last = false; !last && !err;) {
                refill(m, b, gz, lane);
                last = peek(b, 1) != 0;
                const uint32_t type = (peek(b, 3) >> 1) & 3;
                drop(b, 3);
                if (type == 0) {
                    // stored: skip to the byte boundary, LEN, NLEN, LEN raw bytes
                    drop(b, b.cnt & 7);
                    const uint32_t ln = take(m, b, gz, lane, 16), nl = take(m, b, gz, lane, 16);
                    const uint64_t src = consumed(b);
                    if ((ln ^ nl) != 0xFFFFu) err = INF_BAD_BLOCK;
                    else if (src + ln + 8 > in1) err = INF_INPUT_END;
                    else if (op + ln > o1) err = INF_OUTPUT_OVERRUN;
                    else {
                        for (uint32_t j = lane; j < ln; j += 32) out[op + j] = gz[src + j];
                        op += ln;
                        ring_init(m, b, gz, src + ln, lane);
                    }
                    continue;
                }
                if (type == 3) {
                    err = INF_BAD_BLOCK;
                    break;
                }
                if (type == 1) {  // fixed codes (RFC 1951 3.2.6)
                    __syncwarp();
                    for (uint32_t s = lane; s < 288; s += 32) m.len[s] = s < 144 ? 8 : s < 256 ? 9 : s < 280 ? 7 : 8;
                    for (uint32_t s = lane; s < 32; s += 32) m.len[288 + s] = 5;
                    __syncwarp();
                    build_tables<LL_BITS>(m.len, 288, m.ll_cnt, m.ll_sym, m.ll_fast, lane);
                    build_tables<D_BITS>(m.len + 288, 30, m.d_cnt, m.d_sym, m.d_fast, lane);
                } else {  // dynamic codes (3.2.7)
                    const uint32_t hlit = take(m, b, gz, lane, 5) + 257, hdist = take(m, b, gz, lane, 5) + 1;
                    const uint32_t hclen = take(m, b, gz, lane, 4) + 4;
                    if (hlit > 286 || hdist > 30) {
                        err = INF_BAD_BLOCK;
                        break;
                    }
                    __syncwarp();
                    if (lane < 19) m.len[lane] = 0;
                    __syncwarp();
                    for (uint32_t i = 0; i < hclen; ++i) {
                        const uint32_t v = take(m, b, gz, lane, 3);
                        if (lane == 0) m.len[c_clen_order[i]] = (uint8_t)v;
                    }
                    __syncwarp();
                    // the code-length code: 19 symbols, at most 7 bits — its tables borrow the distance arrays
                    if (!build_tables<7>(m.len, 19, m.d_cnt, m.d_sym, m.d_fast, lane)) {
                        err = INF_BAD_CODE;
                        break;
                    }
                    uint32_t i = 0, prev = 0;
                    while (i < hlit + hdist && !err) {
                        refill(m, b, gz, lane);
                        const uint32_t s = decode_sym<7>(b, m.d_fast, m.d_cnt, m.d_sym);
                        uint32_t rep = 1, val = s;
                        if (s < 16) {
                            prev = s;
                        } else if (s == 16) {
                            if (i == 0) err = INF_BAD_CODE;
                            rep = 3 + peek(b, 2);
                            drop(b, 2);
                            val = prev;
                        } else if (s == 17) {
                            rep = 3 + peek(b, 3);
                            drop(b, 3);
                            val = 0;
                            prev = 0;
                        } else if (s == 18) {
                            rep = 11 + peek(b, 7);
                            drop(b, 7);
                            val = 0;
                            prev = 0;
                        } else {
                            err = INF_BAD_CODE;
                        }
                        if (i + rep > hlit + hdist) err = INF_BAD_CODE;
                        if (!err) {
                            // lengths of the literal/length alphabet go to len[0 .. hlit), distances to len[288 ..)
                            for (uint32_t j = lane; j < rep; j += 32) {
                                const uint32_t t = i + j;
                                m.len[t < hlit ? t : 288 + (t - hlit)] = (uint8_t)val;
                            }
                            i += rep;
                        }
                    }
                    if (err) break;
                    __syncwarp();
                    for (uint32_t s = hlit + lane; s < 288; s += 32) m.len[s] = 0;
                    for (uint32_t s = hdist + lane; s < 32; s += 32) m.len[288 + s] = 0;
                    __syncwarp();
                    if (m.len[256] == 0 || !build_tables<LL_BITS>(m.len, 288, m.ll_cnt, m.ll_sym, m.ll_fast, lane) ||
                        !build_tables<D_BITS>(m.len + 288, 30, m.d_cnt, m.d_sym, m.d_fast, lane)) {
                        err = INF_BAD_CODE;
                        break;
                    }
                }
                // ---- symbols of the block ------------------------------------------------------------------------------------------
                for (;;) {
                    refill(m, b, gz, lane);
                    if (consumed(b) > in1) {
                        err = INF_INPUT_END;
                        break;
                    }
                    const uint32_t s = decode_sym<LL_BITS>(b, m.ll_fast, m.ll_cnt, m.ll_sym);
                    if (s < 256) {
                        if (lane == 0) m.lit[n_lit] = (uint8_t)s;
                        if (++n_lit == 64) {
                            __syncwarp();
                            if (op + 64 > o1) {
                                err = INF_OUTPUT_OVERRUN;
                                break;
                            }
                            flush_lits();
                        }
                        continue;
                    }
                    if (s == 256) break;
                    if (s > 285) {
                        err = INF_BAD_CODE;
                        break;
                    }
                    uint32_t len = c_len_base[s - 257] + peek(b, c_len_extra[s - 257]);
                    drop(b, c_len_extra[s - 257]);
                    refill(m, b, gz, lane);
                    const uint32_t ds = decode_sym<D_BITS>(b, m.d_fast, m.d_cnt, m.d_sym);
                    if (ds > 29) {
                        err = INF_BAD_CODE;
                        break;
                    }
                    const uint32_t dist = c_dist_base[ds] + peek(b, c_dist_extra[ds]);
                    drop(b, c_dist_extra[ds]);
                    __syncwarp();
                    if (op + n_lit + len > o1) {
                        err = INF_OUTPUT_OVERRUN;
                        break;
                    }
                    flush_lits();
                    if (dist > op - o0) {
                        err = INF_BAD_DISTANCE;
                        break;
                    }
                    // LZ77 copy: byte k of the match repeats the text `dist` back, with period dist when it overlaps itself
                    const uint8_t* src = out + op - dist;
                    for (uint32_t j = lane; j < len; j += 32) out[op + j] = __ldcg(src + (dist >= len ? j : j % dist));
                    op += len;
                    __syncwarp();
                }
                __syncwarp();
                if (!err) {
                    if (op + n_lit > o1) err = INF_OUTPUT_OVERRUN;
                    else flush_lits();
                }
            }
        }
        // ---- trailer: CRC-32 and ISIZE of the text (RFC 1952 2.3.1) ------------------------------------------------------------------
        if (!err) {
            drop(b, b.cnt & 7);
            const uint64_t t = consumed(b);
            if (t + 8 > in1) err = INF_INPUT_END;
            else if (t + 8 != in1) err = INF_TRAILING;
            else {
                const uint32_t want_crc = gz[t] | gz[t + 1] << 8 | gz[t + 2] << 16 | (uint32_t)gz[t + 3] << 24;
                const uint32_t isize = gz[t + 4] | gz[t + 5] << 8 | gz[t + 6] << 16 | (uint32_t)gz[t + 7] << 24;
                const uint64_t n = op - o0;
                if (op != o1 || (uint32_t)n != isize) err = INF_SIZE_MISMATCH;
                else {
                    // every lane checksums a slice (registers start at zero: pure polynomial remainders), the slices are
                    // combined with crc(A || B) = shift(crc(A), |B|) ^ crc(B); pre/post conditioning is added once at the end
                    __syncwarp();
                    __threadfence_block();
                    const uint64_t per = (n + 31) / 32;
                    const uint64_t a = min(n, per * lane), z = min(n, a + per);
                    uint32_t c = crc_bytes(s_crc_table, out + o0 + a, z - a, 0);
                    uint64_t mylen = z - a;
                    for (int d = 1; d < 32; d <<= 1) {
                        const uint32_t oc = __shfl_down_sync(0xFFFFFFFFu, c, d);
                        const uint64_t ol = __shfl_down_sync(0xFFFFFFFFu, mylen, d);
                        if ((lane & (2 * d - 1)) == 0) {
                            c = crc_shift(c, ol) ^ oc;
                            mylen += ol;
                        }
                    }
                    // crc32(M) = ~rem(x^32 M + init), init contributes shift(0xFFFFFFFF, n)
                    uint32_t crc = ~(c ^ crc_shift(0xFFFFFFFFu, n));
                    crc = __shfl_sync(0xFFFFFFFFu, crc, 0);
                    if (crc != want_crc) err = INF_CRC_MISMATCH;
                }
            }
        }
        if (lane == 0) status[k] = err;
        __syncwarp();
    }
}

}  // namespace gtgpu

using namespace gtgpu;

// Member boundaries of a gzip file on the host: BGZF blocks (an extra field 'B' 'C' carries the block size) are split one
// by one; anything else is ONE member up to the end of the buffer.  Cheap: it touches 18 bytes per member.
extern "C" int32_t gtgpu_gzip_members(const uint8_t* gz, uint64_t n_bytes, uint64_t capacity, uint64_t* out_member_offsets,
                                      uint64_t* out_n_members) try {
    if (!out_n_members || (n_bytes && !gz) || (capacity && !out_member_offsets))
        return fail(GTGPU_ERR_INVALID, "gzip_members: null argument");
    std::vector<uint64_t> offs;
    uint64_t p = 0;
    while (p < n_bytes) {
        offs.push_back(p);
        uint64_t next = n_bytes;  // not BGZF: the rest is one member
        if (p + 18 <= n_bytes && gz[p] == 0x1F && gz[p + 1] == 0x8B && gz[p + 2] == 8 && (gz[p + 3] & 4)) {
            const uint64_t xlen = gz[p + 10] | (uint64_t)gz[p + 11] << 8;
            const uint64_t x_end = std::min(n_bytes, p + 12 + xlen);
            for (uint64_t q = p + 12; q + 4 <= x_end;) {
                const uint64_t slen = gz[q + 2] | (uint64_t)gz[q + 3] << 8;
                if (gz[q] == 'B' && gz[q + 1] == 'C' && slen == 2 && q + 6 <= x_end) {
                    const uint64_t bsize = (gz[q + 4] | (uint64_t)gz[q + 5] << 8) + 1;
                    if (bsize >= 18 && p + bsize <= n_bytes) next = p + bsize;
                    break;
                }
                q += 4 + slen;
            }
        }
        p = next;
    }
    offs.push_back(n_bytes);
    *out_n_members = offs.size() - 1;
    if (offs.size() > capacity) return fail(GTGPU_ERR_CAPACITY, "gzip_members: out_member_offsets needs n_members + 1 entries (count returned)");
    std::copy(offs.begin(), offs.end(), out_member_offsets);
    return GTGPU_OK;
} GT_CATCH

namespace gtgpu {

static void crc_tables(uint32_t* table, uint32_t* pow) {
    for (uint32_t i = 0; i < 256; ++i) {
        uint32_t c = i;
        for (int k = 0; k < 8; ++k) c = (c & 1) ? (c >> 1) ^ 0xEDB88320u : c >> 1;
        table[i] = c;
    }
    auto mul = [](uint32_t a, uint32_t b) {
        uint32_t m = 1u << 31, p = 0;
        for (;;) {
            if (a & m) {
                p ^= b;
                if ((a & (m - 1)) == 0) break;
            }
            m >>= 1;
            b = (b & 1) ? (b >> 1) ^ 0xEDB88320u : b >> 1;
        }
        return p;
    };
    uint32_t p = 1u << 23;  // x^8: one zero byte
    for (int k = 0; k < 32; ++k) {
        pow[k] = p;
        p = mul(p, p);
    }
}

// Device core (the caller holds ctx->mu): d_gz = the members back to back in a 512-byte aligned buffer with >= 2 KiB of
// padding behind them; d_out receives the text.  Synchronises once to read the per-member status.
int32_t gunzip_device(gtgpu_ctx* ctx, uint64_t n_members, const uint8_t* d_gz, const uint64_t* d_member_offsets,
                      const uint64_t* d_out_offsets, uint8_t* d_out, uint32_t* d_status, std::vector<uint32_t>& h_status) {
    static bool tables_on[64] = {false};
    if (ctx->device < 64 && !tables_on[ctx->device]) {
        uint32_t table[256], pow[32];
        crc_tables(table, pow);
        GT_CUDA(cudaMemcpyToSymbol(c_crc_table, table, sizeof table));
        GT_CUDA(cudaMemcpyToSymbol(c_crc_pow, pow, sizeof pow));
        tables_on[ctx->device] = true;
    }
    int occ = 1;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, gunzip_kernel, INF_WARPS * 32, 0) != cudaSuccess || occ < 1) occ = 1;
    const uint64_t blocks = (n_members + INF_WARPS - 1) / INF_WARPS;
    const int grid = (int)std::max<uint64_t>(1, std::min<uint64_t>(blocks, (uint64_t)ctx->sm_count * occ));
    ctx->time_begin();
    gunzip_kernel<<<grid, INF_WARPS * 32, 0, ctx->stream>>>(n_members, d_gz, d_member_offsets, d_out_offsets, d_out, d_status);
    ctx->time_end();
    ctx->launches++;
    GT_CUDA(cudaGetLastError());
    h_status.resize(n_members);
    GT_CUDA(cudaMemcpyAsync(h_status.data(), d_status, n_members * 4, cudaMemcpyDeviceToHost, ctx->stream));
    GT_CUDA(cudaStreamSynchronize(ctx->stream));
    static const char* what[] = {"ok", "bad gzip header", "bad DEFLATE block", "invalid Huffman code", "compressed data ends early",
                                 "more text than the trailer's ISIZE", "distance reaches before the member's text",
                                 "text length differs from ISIZE", "CRC-32 mismatch", "bytes between the last block and the trailer"};
    for (uint64_t k = 0; k < n_members; ++k)
        if (h_status[k])
            return fail(GTGPU_ERR_INVALID, "gunzip: member " + std::to_string(k) + ": " + what[std::min<uint32_t>(h_status[k], 9)]);
    return GTGPU_OK;
}

}  // namespace gtgpu

namespace gtgpu {

// H2D of the members + inflate; the text stays on the device in scratch SC_GZ_OUT (*d_text, *n_text bytes, 64 bytes of
// padding behind it).  The caller holds ctx->mu.  out_member_offsets (host, n_members + 1) may be null.
int32_t gunzip_locked(gtgpu_ctx* ctx, uint64_t n_members, const uint8_t* gz, const uint64_t* member_offsets,
                             uint64_t* out_member_offsets, uint8_t** d_text, uint64_t* n_text) {
    // output size of every member from its trailer (ISIZE, RFC 1952): the text of a member must be < 4 GiB
    std::vector<uint64_t> oo(n_members + 1, 0), rebased(n_members + 1, 0);
    const uint64_t base = n_members ? member_offsets[0] : 0;
    for (uint64_t k = 0; k < n_members; ++k) {
        if (member_offsets[k + 1] < member_offsets[k] + 18)
            return fail(GTGPU_ERR_INVALID, "gunzip: member " + std::to_string(k) + " is shorter than a gzip header + trailer");
        const uint8_t* t = gz + member_offsets[k + 1] - 4;
        oo[k + 1] = oo[k] + (t[0] | (uint64_t)t[1] << 8 | (uint64_t)t[2] << 16 | (uint64_t)t[3] << 24);
        rebased[k + 1] = member_offsets[k + 1] - base;
    }
    if (out_member_offsets) std::copy(oo.begin(), oo.end(), out_member_offsets);
    const uint64_t n_in = rebased[n_members], n_out = oo[n_members];
    *n_text = n_out;
    cudaStream_t st = ctx->stream;
    uint8_t *d_gz, *d_out;
    uint64_t *d_mo, *d_oo;
    uint32_t* d_status;
    GT_TRY(ctx->scratch_get(SC_GZ_IN, n_in + 4096, (void**)&d_gz));
    GT_TRY(ctx->scratch_get(SC_GZ_OUT, n_out + 64, (void**)&d_out));
    GT_TRY(ctx->scratch_get(SC_GZ_MOFF, (n_members + 1) * 8, (void**)&d_mo));
    GT_TRY(ctx->scratch_get(SC_GZ_OOFF, (n_members + 1) * 8, (void**)&d_oo));
    GT_TRY(ctx->scratch_get(SC_GZ_STATUS, n_members * 4 + 4, (void**)&d_status));
    *d_text = d_out;
    if (n_members == 0) return GTGPU_OK;
    GT_CUDA(cudaMemcpyAsync(d_gz, gz + base, n_in, cudaMemcpyHostToDevice, st));
    GT_CUDA(cudaMemsetAsync(d_gz + n_in, 0, 4096, st));
    GT_CUDA(cudaMemsetAsync(d_out + n_out, 0, 64, st));
    GT_CUDA(cudaMemcpyAsync(d_mo, rebased.data(), (n_members + 1) * 8, cudaMemcpyHostToDevice, st));
    GT_CUDA(cudaMemcpyAsync(d_oo, oo.data(), (n_members + 1) * 8, cudaMemcpyHostToDevice, st));
    GT_CUDA(cudaStreamSynchronize(st));  // the offset vectors are pageable
    std::vector<uint32_t> h_status;
    return gunzip_device(ctx, n_members, d_gz, d_mo, d_oo, d_out, d_status, h_status);
}

// gzip members -> device text (SC_GZ_OUT); a text that does not fit in device memory is reported as such
int32_t inflate_whole_locked(gtgpu_ctx* ctx, uint64_t n_members, const uint8_t* gz, const uint64_t* member_offsets, const std::string& who,
                             uint8_t** d_text, uint64_t* n_text, uint64_t* out_member_offsets) {
    const int32_t s = gunzip_locked(ctx, n_members, gz, member_offsets, out_member_offsets, d_text, n_text);
    if (s == GTGPU_ERR_NOMEM)
        return fail(s, who + ": the inflated text does not fit in device memory (gzip input is inflated whole before it is parsed): " +
                           gtgpu_last_error());
    return s;
}

int32_t check_members(uint64_t n_members, const uint8_t* gz, const uint64_t* member_offsets, const char* who) {
    if (n_members && (!gz || !member_offsets)) return fail(GTGPU_ERR_INVALID, std::string(who) + ": null argument");
    for (uint64_t k = 0; k < n_members; ++k)
        if (member_offsets[k] > member_offsets[k + 1]) return fail(GTGPU_ERR_INVALID, std::string(who) + ": member_offsets not monotone");
    return GTGPU_OK;
}

}  // namespace gtgpu

extern "C" int32_t gtgpu_gunzip(gtgpu_ctx* ctx, uint64_t n_members, const uint8_t* gz, const uint64_t* member_offsets,
                                gtgpu_buf** out_text, uint64_t* out_member_offsets) try {
    if (!ctx || !out_text || !out_member_offsets) return fail(GTGPU_ERR_INVALID, "gunzip: null argument");
    GT_TRY(check_members(n_members, gz, member_offsets, "gunzip"));
    std::lock_guard<std::mutex> lk(ctx->mu);
    GT_CUDA(cudaSetDevice(ctx->device));
    uint8_t* d_text = nullptr;
    uint64_t n_text = 0;
    GT_TRY(gunzip_locked(ctx, n_members, gz, member_offsets, out_member_offsets, &d_text, &n_text));
    BufPtr buf;
    const int32_t s = buf_from_device(ctx, d_text, n_text, 1, ctx->stream, &buf);
    if (s == GTGPU_ERR_CUDA) return fail(s, std::string("gunzip: D2H: ") + gtgpu_last_error());
    GT_TRY(s);
    const cudaError_t e = cudaStreamSynchronize(ctx->stream);
    if (e != cudaSuccess) return fail(GTGPU_ERR_CUDA, std::string("gunzip: D2H: ") + cudaGetErrorString(e));
    *out_text = buf.release();
    return GTGPU_OK;
} GT_CATCH

// gtgpu_tokenize_bed on gzip members: inflate on the device, parse + sort + tokenize the text where it is.
extern "C" int32_t gtgpu_tokenize_bed_gz(gtgpu_index* ix, uint64_t n_members, const uint8_t* gz, const uint64_t* member_offsets,
                                         uint32_t n_names, const char* names, const uint32_t* name_offsets, uint32_t unk_id,
                                         gtgpu_buf** out_ids) try {
    if (!ix || !out_ids || (n_names && (!names || !name_offsets))) return fail(GTGPU_ERR_INVALID, "tokenize_bed_gz: null argument");
    GT_TRY(check_members(n_members, gz, member_offsets, "tokenize_bed_gz"));
    gtgpu_ctx* ctx = ix->ctx;
    std::lock_guard<std::mutex> lk(ctx->mu);
    GT_CUDA(cudaSetDevice(ctx->device));
    uint8_t* d_text = nullptr;
    uint64_t n_text = 0;
    GT_TRY(gunzip_locked(ctx, n_members, gz, member_offsets, nullptr, &d_text, &n_text));
    return tokenize_bed_locked(ix, nullptr, (const char*)d_text, n_text, n_names, names, name_offsets, unk_id, out_ids);
} GT_CATCH

// gtgpu_tokenize_fragments_text on gzip members (a bgzip'ed fragment file: thousands of members).  *out_text returns the
// inflated text as well: the barcode spans index into it.  Errors carry the text form's name and messages.
extern "C" int32_t gtgpu_tokenize_fragments_gz(gtgpu_index* ix, uint64_t n_members, const uint8_t* gz, const uint64_t* member_offsets,
                                               uint32_t n_names, const char* names, const uint32_t* name_offsets, uint32_t unk_id,
                                               uint32_t* out_n_barcodes, gtgpu_buf** out_barcode_spans,
                                               gtgpu_buf** out_barcode_offsets, gtgpu_buf** out_ids, gtgpu_buf** out_text) try {
    if (!ix || !out_n_barcodes || !out_barcode_spans || !out_barcode_offsets || !out_ids || !out_text ||
        (n_names && (!names || !name_offsets)))
        return fail(GTGPU_ERR_INVALID, "tokenize_fragments_gz: null argument");
    GT_TRY(check_members(n_members, gz, member_offsets, "tokenize_fragments_gz"));
    gtgpu_ctx* ctx = ix->ctx;
    std::lock_guard<std::mutex> lk(ctx->mu);
    GT_CUDA(cudaSetDevice(ctx->device));
    uint8_t* d_text = nullptr;
    uint64_t n_text = 0;
    GT_TRY(gunzip_locked(ctx, n_members, gz, member_offsets, nullptr, &d_text, &n_text));
    if (n_text >= 0xFFFFFFF0ull) return fail(GTGPU_ERR_UNSUPPORTED, "tokenize_fragments_text: at most 4 GiB of text per call");
    BufPtr text, spans, offs, ids;  // the text's copy on copy_out overlaps the parse
    int32_t s = buf_from_device(ctx, d_text, n_text, 1, ctx->copy_out, &text);
    if (s == GTGPU_ERR_CUDA) return fail(s, "tokenize_fragments_gz: D2H of the text failed");
    GT_TRY(s);
    try {
        s = tokenize_fragments_file_locked(ix, nullptr, (const char*)d_text, n_text, n_names, names, name_offsets, unk_id,
                                           "tokenize_fragments_text", out_n_barcodes, nullptr, nullptr, &spans, &offs, &ids);
    } catch (...) {
        cudaStreamSynchronize(ctx->copy_out);  // the text's copy ends before its block goes back to the cache
        throw;
    }
    if (s == GTGPU_OK && cudaStreamSynchronize(ctx->copy_out) != cudaSuccess) s = fail(GTGPU_ERR_CUDA, "tokenize_fragments_gz: D2H of the text failed");
    if (s != GTGPU_OK) {
        cudaStreamSynchronize(ctx->copy_out);
        return s;
    }
    *out_barcode_spans = spans.release();
    *out_barcode_offsets = offs.release();
    *out_ids = ids.release();
    *out_text = text.release();
    return GTGPU_OK;
} GT_CATCH

// gtgpu_tokenize_fragments_file on gzip members: inflated whole into device memory, then tokenized in windows where it is.
extern "C" int32_t gtgpu_tokenize_fragments_file_gz(gtgpu_index* ix, uint64_t n_members, const uint8_t* gz, const uint64_t* member_offsets,
                                                    uint32_t n_names, const char* names, const uint32_t* name_offsets, uint32_t unk_id,
                                                    uint32_t* out_n_barcodes, gtgpu_buf** out_barcode_names,
                                                    gtgpu_buf** out_barcode_name_offsets, gtgpu_buf** out_barcode_offsets,
                                                    gtgpu_buf** out_ids) try {
    if (!ix || !out_n_barcodes || !out_barcode_names || !out_barcode_name_offsets || !out_barcode_offsets || !out_ids ||
        (n_names && (!names || !name_offsets)))
        return fail(GTGPU_ERR_INVALID, "tokenize_fragments_file_gz: null argument");
    GT_TRY(check_members(n_members, gz, member_offsets, "tokenize_fragments_file_gz"));
    gtgpu_ctx* ctx = ix->ctx;
    std::lock_guard<std::mutex> lk(ctx->mu);
    GT_CUDA(cudaSetDevice(ctx->device));
    uint8_t* d_text = nullptr;
    uint64_t n_text = 0;
    GT_TRY(inflate_whole_locked(ctx, n_members, gz, member_offsets, "tokenize_fragments_file_gz", &d_text, &n_text));
    BufPtr nm, no, offs, ids;
    GT_TRY(tokenize_fragments_file_locked(ix, nullptr, (const char*)d_text, n_text, n_names, names, name_offsets, unk_id,
                                          "tokenize_fragments_file_gz", out_n_barcodes, &nm, &no, nullptr, &offs, &ids));
    *out_barcode_names = nm.release();
    *out_barcode_name_offsets = no.release();
    *out_barcode_offsets = offs.release();
    *out_ids = ids.release();
    return GTGPU_OK;
} GT_CATCH
