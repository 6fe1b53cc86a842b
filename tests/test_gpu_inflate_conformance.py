"""gtgpu_gunzip against zlib at every DEFLATE construct the device inflater has its own code for.

The streams come from a bit-level DEFLATE writer in this file: stored, fixed and dynamic blocks from explicit token lists,
with chosen code lengths for the three alphabets, chosen run-length coding of those lengths and raw bit fields for invalid
streams, wrapped in gzip members with optional FEXTRA / FNAME / FCOMMENT / FHCRC.  Every stream is checked against zlib on
the host first (the tests without the gpu mark), so a writer mistake cannot pass for a decoder mistake.  On the device each
valid case must give zlib's text and member offsets, once as its own member and once among all cases in one call; each
invalid case must fail with the reason of its first problem, alone and as member 1 between two good members.

Incomplete Huffman codes follow zlib's inflate: a literal/length or distance code may hold no code or a single 1-bit code;
any other incomplete set, a single code of two or more bits included, is an invalid stream."""
import bisect
import gzip
import random
import re
import struct
import zlib

import numpy as np
import pytest

LEN_BASE = [3, 4, 5, 6, 7, 8, 9, 10, 11, 13, 15, 17, 19, 23, 27, 31, 35, 43, 51, 59, 67, 83, 99, 115, 131, 163, 195, 227, 258]
LEN_EXTRA = [0] * 8 + [1] * 4 + [2] * 4 + [3] * 4 + [4] * 4 + [5] * 4 + [0]
LEN_MAX = [b + (1 << e) - 1 for b, e in zip(LEN_BASE, LEN_EXTRA)]
LEN_MAX[27] = 257  # symbol 284 covers 227..257 (RFC 1951 3.2.5); 258 is symbol 285
DIST_BASE = [1, 2, 3, 4, 5, 7, 9, 13, 17, 25, 33, 49, 65, 97, 129, 193, 257, 385, 513, 769, 1025, 1537, 2049, 3073, 4097, 6145,
             8193, 12289, 16385, 24577]
DIST_EXTRA = [0, 0, 0, 0] + [k // 2 for k in range(2, 28)]
DIST_MAX = [b + (1 << e) - 1 for b, e in zip(DIST_BASE, DIST_EXTRA)]
CLEN_ORDER = [16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15]
FIXED_LL = [8] * 144 + [9] * 112 + [7] * 24 + [8] * 8
FIXED_D = [5] * 32

# the reasons gunzip_device reports, by status
BAD_HEADER, BAD_BLOCK, BAD_CODE = "bad gzip header", "bad DEFLATE block", "invalid Huffman code"
INPUT_END, OVERRUN, BAD_DIST = "compressed data ends early", "more text than the trailer's ISIZE", "distance reaches before the member's text"
SIZE, CRC, TRAILING = "text length differs from ISIZE", "CRC-32 mismatch", "bytes between the last block and the trailer"
SHORT = "is shorter than a gzip header + trailer"


# ---- a DEFLATE writer (RFC 1951) --------------------------------------------------------------------------------------------
class BitWriter:
    def __init__(self):
        self.out, self.acc, self.n = bytearray(), 0, 0

    def bits(self, v, n):
        """n bits of v, least significant first (RFC 1951 3.1.1)"""
        self.acc |= (v & ((1 << n) - 1)) << self.n
        self.n += n
        while self.n >= 8:
            self.out.append(self.acc & 0xFF)
            self.acc >>= 8
            self.n -= 8

    def code(self, c, n):
        """a Huffman code: most significant bit first"""
        self.bits(int(format(c & ((1 << n) - 1), f"0{n}b")[::-1], 2), n)

    def align(self):
        self.bits(0, -self.n % 8)

    def raw(self, data):
        assert self.n == 0
        self.out += data

    def getvalue(self):
        self.align()
        return bytes(self.out)


def canonical(lengths):
    """Canonical codes of a list of code lengths (RFC 1951 3.2.2); None for length 0."""
    count = [0] * 16
    for n in lengths:
        count[n] += 1
    count[0] = 0
    nxt, code = [0] * 16, 0
    for n in range(1, 16):
        code = (code + count[n - 1]) << 1
        nxt[n] = code
    out = []
    for n in lengths:
        out.append(nxt[n] if n else None)
        nxt[n] += bool(n)
    return out


def kraft_gap(lengths: dict, maxbits=15):
    return (1 << maxbits) - sum(1 << (maxbits - n) for n in lengths.values())


def complete(lengths: dict, spare, maxbits=15):
    """Gives spare symbols the lengths that make the Kraft sum of `lengths` exactly 1."""
    gap = kraft_gap(lengths, maxbits)
    assert 0 <= gap < 1 << maxbits
    spare = iter(s for s in spare if s not in lengths)
    for b in range(maxbits):
        if gap >> b & 1:
            lengths[next(spare)] = maxbits - b
    return lengths


def balanced(symbols):
    """A complete code over exactly these symbols, lengths d - 1 and d; a single symbol gets one 1-bit code."""
    symbols = sorted(symbols)
    if len(symbols) == 1:
        return {symbols[0]: 1}
    d = (len(symbols) - 1).bit_length()
    short = (1 << d) - len(symbols)
    return {s: d - 1 if i < short else d for i, s in enumerate(symbols)}


def deep(symbols, rng, maxbits=15):
    """Random lengths of 1..maxbits bits for the symbols: many codes longer than the decoder's first-level tables.  The
    Kraft sum is made exactly 1 by shortening the shortest codes whose weight is at most the lowest bit of the gap (one
    always is)."""
    if len(symbols) == 1:
        return balanced(symbols)
    out, cap = {}, 1 << maxbits
    syms = sorted(symbols)
    rng.shuffle(syms)
    for k, s in enumerate(syms):
        rest = len(syms) - k - 1
        n = rng.choice([n for n in range(1, maxbits + 1) if cap - (1 << (maxbits - n)) >= rest])
        out[s] = n
        cap -= 1 << (maxbits - n)
    while cap:
        low = cap & -cap
        s = min((s for s in syms if 1 << (maxbits - out[s]) <= low), key=lambda s: out[s])
        cap -= 1 << (maxbits - out[s])
        out[s] -= 1
    return out


def len_symbol(n):
    assert 3 <= n <= 258
    i = 28 if n == 258 else bisect.bisect_right(LEN_BASE, n) - 1
    return 257 + i, n - LEN_BASE[i], LEN_EXTRA[i]


def dist_symbol(d):
    i = bisect.bisect_right(DIST_BASE, d) - 1
    return i, d - DIST_BASE[i], DIST_EXTRA[i]


def used_symbols(tokens):
    ll, d = {256}, set()
    for t in tokens:
        if isinstance(t, int):
            ll.add(t)
        elif isinstance(t[0], int):
            ll.add(len_symbol(t[0])[0])
            d.add(dist_symbol(t[1])[0])
    return ll, d


def run_lengths(seq):
    """Greedy run-length coding of code lengths with 16 / 17 / 18, across the literal/length - distance boundary."""
    out, i = [], 0
    while i < len(seq):
        v, j = seq[i], i
        while j < len(seq) and seq[j] == v:
            j += 1
        n = j - i
        if v == 0:
            while n >= 3:
                k = min(n, 138)
                out.append((18, k) if k >= 11 else (17, k))
                n -= k
            out += [0] * n
        else:
            out.append(v)
            n -= 1
            while n >= 3:
                k = min(n, 6)
                out.append((16, k))
                n -= k
            out += [v] * n
        i = j
    return out


def expand(rle):
    out = []
    for it in rle:
        if isinstance(it, int):
            out.append(it)
        else:
            out += [out[-1] if it[0] == 16 else 0] * it[1]
    return out


class Deflate:
    """A raw DEFLATE stream and the text it decodes to.  Tokens: an int is a literal, (length, distance) a match,
    ("ll", sym) a bare literal/length symbol, ("d", length, dsym) a match with a bare distance symbol."""

    def __init__(self):
        self.w, self.text = BitWriter(), bytearray()

    def header(self, last, btype):
        self.w.bits(int(last), 1)
        self.w.bits(btype, 2)
        return self

    def stored(self, data, last=False, ln=None, nln=None):
        self.header(last, 0)
        self.w.align()
        assert ln is not None or len(data) <= 65535
        ln = len(data) if ln is None else ln
        self.w.bits(ln, 16)
        self.w.bits(~ln if nln is None else nln, 16)
        self.w.raw(data)
        self.text += data
        return self

    def fixed(self, tokens, last=False):
        self.header(last, 1)
        self.symbols(tokens, FIXED_LL, FIXED_D)
        return self

    def dynamic(self, tokens, last=False, ll=None, d=None, cl=None, rle=None, hlit=None, hdist=None, hclen=None, eob=True,
                strict=True):
        """ll / d / cl: {symbol: code length} (default: a balanced code over the used symbols); rle: the code-length
        symbols, ints 0..15 and (16|17|18, count) (default: run_lengths; "plain": one symbol per length)."""
        u_ll, u_d = used_symbols(tokens)
        ll = balanced(u_ll if eob else u_ll - {256}) if ll is None else ll
        d = (balanced(u_d) if u_d else {}) if d is None else d
        hlit = hlit or max(max(ll, default=0) + 1, 257)
        hdist = hdist or max(max(d, default=0) + 1, 1)
        seq = [ll.get(s, 0) for s in range(hlit)] + [d.get(s, 0) for s in range(hdist)]
        rle = run_lengths(seq) if rle is None else list(seq) if rle == "plain" else rle
        if strict:
            assert expand(rle) == seq
        cl = balanced({it if isinstance(it, int) else it[0] for it in rle}) if cl is None else cl
        hclen = hclen or max(4, max(CLEN_ORDER.index(s) + 1 for s in cl if cl[s]))
        self.header(last, 2)
        self.w.bits(hlit - 257, 5)
        self.w.bits(hdist - 1, 5)
        self.w.bits(hclen - 4, 4)
        for s in CLEN_ORDER[:hclen]:
            self.w.bits(cl.get(s, 0), 3)
        cls = [cl.get(s, 0) for s in range(19)]
        codes = canonical(cls)
        for it in rle:
            s, n = (it, 0) if isinstance(it, int) else it
            self.w.code(codes[s], cls[s])
            if s >= 16:
                self.w.bits(n - (3, 3, 11)[s - 16], (2, 3, 7)[s - 16])
        self.symbols(tokens, [ll.get(s, 0) for s in range(288)], [d.get(s, 0) for s in range(32)], eob)
        return self

    def symbols(self, tokens, ll, d, eob=True):
        llc, dc = canonical(ll), canonical(d)
        for t in tokens:
            if isinstance(t, int):
                self.w.code(llc[t], ll[t])
                self.text.append(t)
            elif t[0] == "ll":
                self.w.code(llc[t[1]], ll[t[1]])
            else:
                n = t[1] if t[0] == "d" else t[0]
                s, e, ne = len_symbol(n)
                self.w.code(llc[s], ll[s])
                self.w.bits(e, ne)
                if t[0] == "d":
                    self.w.code(dc[t[2]], d[t[2]])
                    continue
                ds, de, dne = dist_symbol(t[1])
                self.w.code(dc[ds], d[ds])
                self.w.bits(de, dne)
                if t[1] <= len(self.text):
                    for _ in range(n):
                        self.text.append(self.text[-t[1]])
        if eob:
            self.w.code(llc[256], ll[256])

    def raw(self):
        return self.w.getvalue()

    def member(self, **kw):
        return member(self.raw(), bytes(self.text), **kw), bytes(self.text)


def member(deflate, text, *, flg=0, extra=None, name=None, comment=None, hcrc=False, cm=8, crc=None, isize=None):
    """A gzip member (RFC 1952) around a raw DEFLATE stream."""
    f = flg | (4 if extra is not None else 0) | (8 if name is not None else 0) | (16 if comment is not None else 0) | (2 if hcrc else 0)
    h = bytes([0x1F, 0x8B, cm, f]) + b"\0\0\0\0\x00\xff"
    if extra is not None:
        h += struct.pack("<H", len(extra)) + extra
    if name is not None:
        h += name + b"\0"
    if comment is not None:
        h += comment + b"\0"
    if hcrc:
        h += struct.pack("<H", zlib.crc32(h) & 0xFFFF)
    crc = zlib.crc32(text) if crc is None else crc
    return h + deflate + struct.pack("<II", crc, (len(text) if isize is None else isize) & 0xFFFFFFFF)


def zlib_inflate(m):
    """zlib's text of ONE member, or None when zlib rejects it (zlib.decompress would stop after a first member)."""
    d = zlib.decompressobj(31)
    try:
        out = d.decompress(m) + d.flush()
    except zlib.error:
        return None
    return out if d.eof and not d.unused_data else None


# ---- valid streams ----------------------------------------------------------------------------------------------------------
def random_tokens(rng, n, alphabet, dist_codes=range(30), max_len=258, p_match=0.3, size=0):
    toks = []
    for _ in range(n):
        codes = [c for c in dist_codes if DIST_BASE[c] <= size]
        if codes and rng.random() < p_match:
            c = rng.choice(codes)
            ln = rng.randint(3, max_len)
            toks.append((ln, rng.randint(DIST_BASE[c], min(DIST_MAX[c], size))))
            size += ln
        else:
            toks.append(rng.choice(alphabet))
            size += 1
    return toks


def deep_block(d: Deflate, rng, tokens, last=False):
    """A dynamic block whose trees take random lengths up to 15 bits."""
    u_ll, u_d = used_symbols(tokens)
    ll = deep(u_ll, rng)
    dd = deep(u_d, rng) if u_d else {}
    return d.dynamic(tokens, last, ll=ll, d=dd)


def tree_cases():
    rng = random.Random(1)
    out = {}
    # literal/length lengths 1..15: 14 literals at 1..14 bits, end-of-block and length 3 at 15; distance codes at 1..15 bits
    letters = list(b"ABCDEFGHIJKLMN")
    ll = {s: k + 1 for k, s in enumerate(letters)} | {256: 15, 257: 15}
    dd = {c: c + 1 for c in range(14)} | {14: 15, 15: 15}
    assert kraft_gap(ll) == 0 and kraft_gap(dd) == 0
    lits = letters + [rng.choice(letters) for _ in range(400)]
    toks = lits + [(3, rng.randint(DIST_BASE[c], DIST_MAX[c])) for c in range(16) for _ in range(3)] + letters[::-1]
    out["ll_1_to_15_bits_d_1_to_15_bits"] = Deflate().dynamic(toks, True, ll=ll, d=dd).member()
    for seed in range(8):  # random deep trees: codes of 11-15 bits on the slow path, distances over 9 bits
        r = random.Random(100 + seed)
        toks = random_tokens(r, 3000, r.sample(range(256), 40), dist_codes=r.sample(range(30), 12), size=0)
        out[f"deep_trees_{seed}"] = deep_block(Deflate(), r, toks, last=True).member()
    out["single_1bit_distance_code_0"] = Deflate().dynamic(list(b"abcd") + [(5, 1), (258, 1), 120, (3, 1)], True, d={0: 1}).member()
    out["single_1bit_distance_code_5"] = Deflate().dynamic(list(b"abcdefgh") + [(10, 7), (4, 8)], True, d={5: 1}).member()
    out["no_distance_codes"] = Deflate().dynamic(list(b"literals only, hdist = 1 with a zero length\n"), True).member()
    empty_ll = {256: 1}
    out["end_of_block_only_blocks"] = (Deflate().dynamic([], ll=empty_ll, d={}).fixed([]).fixed(list(b"abc")).dynamic([], ll=empty_ll)
                                       .fixed([], last=True).member())
    out["end_of_block_only_member"] = Deflate().dynamic([], True, ll=empty_ll, d={}).member()
    # hlit 286 and hdist 30 with the unused symbols at length 0, every code-length symbol sent (hclen 19)
    toks = random_tokens(rng, 500, list(b"xyz \n"), dist_codes=range(8))
    out["hlit_286_hdist_30_hclen_19"] = Deflate().dynamic(toks, True, hlit=286, hdist=30, hclen=19, rle="plain").member()
    # hclen 5: 16, 17, 18, 0 and 8, the least that can give a length other than 0 (hclen 4 is in the invalid cases)
    ll = {s: 8 for s in range(255)} | {256: 8}
    out["hclen_5"] = Deflate().dynamic(list(range(255)) + list(b"hclen"), True, ll=ll, d={}).member()
    # every repeat at its minimum and maximum count; an 18 that runs from the literal/length lengths into the distance ones
    ll = {s: 8 for s in range(149, 160)} | {256: 1, 257: 2, 258: 3, 259: 4, 260: 6, 261: 8}
    dd = {5: 2, 6: 2, 7: 2, 8: 2}
    rle = [(18, 138), (18, 11), 8, (16, 6), 8, (16, 3), (17, 3), (17, 10), (18, 83), 1, 2, 3, 4, 6, 8, (18, 29), 2, (16, 3)]
    lits = [rng.randint(149, 159) for _ in range(40)]
    toks = lits + [(ln, rng.randint(7, 24)) for ln in range(3, 8) for _ in range(4)] + lits
    out["repeats_min_max_and_across"] = Deflate().dynamic(toks, True, ll=ll, d=dd, rle=rle, hlit=286, hdist=9).member()
    # a 16 whose repeats run from the literal/length lengths into the distance lengths
    ll = {s: 9 for s in range(256)} | {256: 2, 257: 2}
    dd = {0: 2, 1: 2, 2: 2, 3: 2}
    d = Deflate()
    toks = list(b"sixteen across ") + [(3, 1), (3, 2), (3, 3), (3, 4)]
    d.dynamic(toks, True, ll=ll, d=dd)
    assert run_lengths([9] * 256 + [2, 2, 2, 2, 2, 2])[-2:] == [2, (16, 5)]
    out["repeat_16_across"] = d.member()
    return out


def match_cases():
    rng = random.Random(2)
    out = {}
    pre = [rng.choice(b"ACGT\t\n0123456789") for _ in range(300)]
    ext = [(ln, rng.randint(1, 300)) for lo, hi in zip(LEN_BASE, LEN_MAX) for ln in (lo, hi)]
    out["length_symbols_extremes_fixed"] = Deflate().fixed(pre + ext, True).member()
    out["length_symbols_extremes_dynamic"] = Deflate().dynamic(pre + ext[::-1], True).member()
    out["every_length_3_to_258"] = Deflate().dynamic(pre + [(ln, rng.randint(1, 300)) for ln in range(3, 259)], True).member()
    far = bytes(rng.randrange(256) for _ in range(40_000))
    dists = [(rng.randint(3, 258), dd) for lo, hi in zip(DIST_BASE, DIST_MAX) for dd in (lo, hi)]
    assert dists[-1][1] == 32768
    out["distance_codes_extremes_fixed"] = Deflate().stored(far).fixed(dists, True).member()
    out["distance_codes_extremes_dynamic"] = Deflate().stored(far[:20_000]).stored(far[20_000:]).dynamic(dists[::-1], True).member()
    out["distance_codes_extremes_deep"] = deep_block(Deflate().stored(far), rng, dists, last=True).member()
    toks = [rng.choice(b"ab") for _ in range(40)]
    for dd in range(1, 41):  # copies that overlap themselves: 32 <= distance < length is one lane round per period
        toks += [(ln, dd) for ln in sorted({3, dd - 1, dd, dd + 1, 2 * dd + 1, 258} - {0, 1, 2})] + [rng.choice(b"xyz")]
    out["overlapping_copies_fixed"] = Deflate().fixed(toks, True).member()
    out["overlapping_copies_dynamic"] = Deflate().dynamic(toks, True).member()
    for k in (1, 2, 31, 32, 33, 100, 258, 1000):  # the copy reaches exactly back to the member's first byte
        lits = [rng.choice(b"0123456789") for _ in range(k)]
        out[f"distance_equals_text_{k}"] = Deflate().fixed(lits + [(min(258, k + 7), k)], True).member()
    out["distance_equals_text_after_stored"] = Deflate().stored(far[:5000]).dynamic([(258, 5000)], True).member()
    return out


def literal_run_cases():
    rng = random.Random(3)
    out = {}
    for n in (63, 64, 65, 127, 128, 129):  # the 64-byte literal buffer flushes at 64
        run = [rng.randrange(256) for _ in range(n)]
        toks = run + [(5, n)] + run + [(n % 50 + 3, 7)] + run
        out[f"literal_run_{n}_fixed"] = Deflate().fixed(toks).fixed(run, True).member()
        out[f"literal_run_{n}_dynamic"] = Deflate().dynamic(toks).dynamic(run, True).member()
    return out


def stored_cases():
    rng = random.Random(4)
    out = {}
    big = bytes(rng.randrange(256) for _ in range(65535))
    out["stored_len_0_mid_member"] = Deflate().fixed(list(b"abc")).stored(b"").fixed(list(b"def") + [(6, 6)]).stored(b"", True).member()
    out["stored_len_1"] = Deflate().stored(b"x").fixed([(10, 1)]).stored(b"y", True).member()
    out["stored_len_65535"] = Deflate().stored(big).fixed([(258, 32768)]).stored(big, True).member()
    out["stored_only_first_and_last"] = Deflate().stored(b"first ").dynamic(list(b"middle ") + [(4, 7)]).stored(b"last", True).member()
    out["stored_several_in_a_row"] = (Deflate().stored(big[:1000]).stored(big[1000:1001]).stored(b"").stored(big[1001:5000])
                                      .stored(big[5000:5513], True).member())
    for phase in range(8):  # the compressed block before the stored one ends at every bit phase: 10 + 9 k bits
        d = Deflate().fixed([144 + (k * 7) % 112 for k in range((phase - 2) % 8)] + list(b"0123"))
        assert d.w.n == (phase + 32) % 8  # four 8-bit literals shift nothing
        out[f"stored_after_bit_phase_{phase}"] = d.stored(big[:300]).fixed([(200, 250)], True).member()
    return out


def ring_cases():
    """Block headers and stored payloads at every byte offset around the 512-byte segments and the 1 KiB ring."""
    rng = random.Random(5)
    out = {}
    pay = bytes(rng.randrange(256) for _ in range(70_000))
    tail = random_tokens(rng, 400, list(b"ACGT\t\n"), size=60)
    targets = [*range(496, 530), *range(1008, 1042), *range(1520, 1538), *range(2032, 2066), 4095, 4096, 4097, 40_001, 65_550]
    for t in targets:  # as its own member at offset 0: the stored payload starts at byte 15, the next block at t
        d = Deflate().stored(pay[:t - 15])
        assert len(d.raw()) + 10 == t
        r = random.Random(t)
        out[f"ring_block_header_at_{t}"] = deep_block(d, r, tail[: r.randint(1, len(tail))]).fixed(tail[:50], True).member()
    for t in (1020, 1023, 1024, 1025, 1030, 2047, 2048, 2049, 3000):  # the first block behind a long FNAME / FCOMMENT
        d = Deflate().dynamic(tail, True)
        key = "name" if t % 2 else "comment"
        m, text = d.member(**{key: b"n" * (t - 11)})
        assert m[t:t + len(d.raw())] == d.raw()
        out[f"ring_first_block_behind_{key}_at_{t}"] = m, text
    m, text = Deflate().fixed(tail, True).member(extra=b"XY" + struct.pack("<H", 1200) + b"e" * 1200, name=b"f.bed", comment=b"c",
                                                 hcrc=True)
    out["ring_every_header_field"] = m, text
    return out


def bed_text(rng, n_lines):
    return "".join(f"chr{rng.randint(1, 22)}\t{a}\t{a + rng.randint(1, 900)}\tname{a % 97}\t{a % 1000}\t+\n"
                   for a in (rng.randint(0, 200_000_000) for _ in range(n_lines))).encode()


def zlib_cases():
    rng = random.Random(6)
    out = {}
    text = bed_text(rng, 4000)

    def gz(level=6, wbits=15, mem=8, strategy=zlib.Z_DEFAULT_STRATEGY, flush=None, every=None):
        co = zlib.compressobj(level, zlib.DEFLATED, 16 + wbits, mem, strategy)
        if flush is None:
            return co.compress(text) + co.flush(), text
        return b"".join(co.compress(text[a:a + every]) + co.flush(flush) for a in range(0, len(text), every)) + co.flush(), text

    for name in ("Z_FILTERED", "Z_HUFFMAN_ONLY", "Z_RLE", "Z_FIXED"):
        out[f"zlib_{name}"] = gz(strategy=getattr(zlib, name))
    for mem in (1, 9):
        out[f"zlib_memlevel_{mem}"] = gz(mem=mem)
    for wbits in range(9, 16):
        out[f"zlib_wbits_{wbits}"] = gz(level=9, wbits=wbits)
    for flush in ("Z_SYNC_FLUSH", "Z_FULL_FLUSH"):
        for every in (1, 700, 65536):
            out[f"zlib_{flush}_every_{every}"] = gz(flush=getattr(zlib, flush), every=every) if every > 1 else \
                gz(flush=getattr(zlib, flush), every=997)
    return out


def size_cases():
    """CRC-32 slices: every length to 300 (lanes with empty slices), and 32 k - 1, 32 k, 32 k + 1."""
    rng = random.Random(7)
    out = {}
    pool = bed_text(rng, 3000)
    for n in range(301):
        t = pool[n * 7:n * 7 + n]
        out[f"text_length_{n}"] = gzip.compress(t, compresslevel=(6, 0, 1)[n % 3], mtime=0), t
    for k in (1, 2, 3, 33, 1000, 2049):
        for n in (32 * k - 1, 32 * k, 32 * k + 1):
            t = pool[:n]
            out[f"text_length_{n}"] = gzip.compress(t, compresslevel=6, mtime=0), t
    return out


def valid_cases():
    out = {}
    for f in (tree_cases, match_cases, literal_run_cases, stored_cases, ring_cases, zlib_cases, size_cases):
        out.update(f())
    return out


# ---- invalid streams --------------------------------------------------------------------------------------------------------
def invalid_cases():
    """name -> (member, reason of its first problem)"""
    rng = random.Random(8)
    out = {}
    lits = list(b"an invalid stream, with a few matches. ")
    toks = lits + [(5, 4), (9, 30), (20, 2)] + lits
    u_ll, u_d = used_symbols(toks)
    text = Deflate().fixed(toks, True).text

    def dyn(**kw):
        last = kw.pop("tokens", toks)
        return member(Deflate().dynamic(last, True, **kw).raw(), text)

    out["block_type_3"] = member(Deflate().header(True, 3).raw() + bytes(16), b""), BAD_BLOCK
    for h in (287, 288):
        out[f"hlit_{h}"] = dyn(hlit=h), BAD_BLOCK
    for h in (31, 32):
        out[f"hdist_{h}"] = dyn(hdist=h), BAD_BLOCK
    out["hclen_4_no_length_can_be_set"] = member(Deflate().dynamic([], True, ll={}, d={}, cl={18: 1, 0: 1}, hlit=257, hdist=1, hclen=4,
                                                                   eob=False).raw(), b""), BAD_CODE
    seq_rle = run_lengths([balanced(u_ll).get(s, 0) for s in range(max(u_ll) + 1)] + [balanced(u_d).get(s, 0) for s in range(max(u_d) + 1)])
    cl = balanced({it if isinstance(it, int) else it[0] for it in seq_rle})
    out["code_length_code_over_subscribed"] = dyn(cl=cl | {next(s for s in range(19) if s not in cl): 1}), BAD_CODE
    short = min(cl, key=lambda s: (cl[s], s))
    out["code_length_code_incomplete"] = dyn(cl=cl | {short: cl[short] + 1}), BAD_CODE
    ll = balanced(u_ll)
    out["literal_length_code_over_subscribed"] = dyn(ll=ll | {255: 1}), BAD_CODE
    out["literal_length_code_incomplete"] = dyn(ll=ll | {256: ll[256] + 1}), BAD_CODE
    assert len(u_d) == 3
    out["distance_code_incomplete"] = dyn(d={c: 2 for c in u_d}), BAD_CODE
    # one distance code of 2 bits: zlib's inflate rejects it (only a 1-bit single code is allowed)
    out["single_2bit_distance_code"] = member(Deflate().dynamic(lits + [(4, 1)], True, d={0: 2}).raw(), bytes(lits) + bytes(lits[-1:]) * 4), BAD_CODE
    out["no_end_of_block_code"] = member(Deflate().dynamic(lits, True, eob=False).raw() + bytes(4), bytes(lits)), BAD_CODE
    seq = [ll.get(s, 0) for s in range(max(ll) + 1)] + [balanced(u_d).get(s, 0) for s in range(max(u_d) + 1)]
    rle = run_lengths(seq)
    out["repeat_16_first"] = dyn(rle=[(16, 3)] + rle, strict=False), BAD_CODE
    out["repeat_past_hlit_plus_hdist"] = dyn(rle=run_lengths(seq[:-1]) + [(17, 3)], strict=False), BAD_CODE
    for s in (286, 287):
        out[f"fixed_literal_length_symbol_{s}"] = member(Deflate().fixed(lits + [("ll", s)], True).raw(), bytes(lits)), BAD_CODE
    for s in (30, 31):
        out[f"fixed_distance_symbol_{s}"] = member(Deflate().fixed(lits + [("d", 3, s)], True).raw(), bytes(lits)), BAD_CODE
    for k in (1, 5, 300):  # ISIZE leaves room for the copy, so the distance is the first problem
        lit = [rng.randrange(256) for _ in range(k)]
        out[f"distance_one_past_text_{k}"] = member(Deflate().fixed(lit + [(3, k + 1)], True).raw(), bytes(lit) + bytes(3)), BAD_DIST
    out["distance_one_past_stored_text"] = member(Deflate().stored(b"12345678").fixed([(3, 9)], True).raw(), b"12345678123"), BAD_DIST
    out["stored_len_nlen_differ"] = member(Deflate().stored(b"stored", True, nln=~6 ^ 0x100).raw(), b"stored"), BAD_BLOCK
    out["stored_len_past_member"] = member(Deflate().stored(b"stored", True, ln=30).raw(), b"stored"), INPUT_END
    # cut inside the run of code-length symbols: the last 8 bytes (read as the trailer) are zero, ISIZE 0
    cut = Deflate().dynamic([], True, ll={}, d={}, cl={18: 1, 0: 2, 8: 2}, rle=[(18, 11)] * 28, hlit=286, hdist=30, eob=False,
                            strict=False).raw()
    assert cut[-12:] == bytes(12)
    out["cut_off_inside_dynamic_header"] = member(b"", b"")[:10] + cut[:-4], INPUT_END
    good, gt = Deflate().dynamic(toks, True).member()
    out["byte_between_last_block_and_trailer"] = good[:-8] + b"\0" + good[-8:], TRAILING
    out["isize_one_too_small"] = good[:-4] + struct.pack("<I", len(gt) - 1), OVERRUN
    out["isize_one_too_large"] = good[:-4] + struct.pack("<I", len(gt) + 1), SIZE
    for bit in (0, 31):
        out[f"crc_bit_{bit}_flipped"] = member(Deflate().dynamic(toks, True).raw(), gt, crc=zlib.crc32(gt) ^ (1 << bit)), CRC
    for f in (0x20, 0x40, 0x80):
        out[f"reserved_flag_{f:#x}"] = member(Deflate().fixed(toks, True).raw(), gt, flg=f), BAD_HEADER
    out["cm_7"] = member(Deflate().fixed(toks, True).raw(), gt, cm=7), BAD_HEADER
    # FNAME runs to the member's end (no NUL anywhere behind it, so ISIZE is 0x01010101)
    out["fname_without_nul"] = bytes([0x1F, 0x8B, 8, 8, 0, 0, 0, 0, 0, 0xFF]) + b"name.bed" * 3 + b"\1" * 8, BAD_HEADER
    out["fextra_past_member"] = bytes([0x1F, 0x8B, 8, 4, 0, 0, 0, 0, 0, 0xFF]) + struct.pack("<H", 1000) + b"x" * 12 + bytes(8), BAD_HEADER
    out["shorter_than_18_bytes"] = member(Deflate().fixed([], True).raw(), b"")[:17], SHORT
    return out


# ---- BGZF splitting (host) ---------------------------------------------------------------------------------------------------
def bgzf_member(text, before=b"", after=b"", bsize=None):
    co = zlib.compressobj(6, zlib.DEFLATED, -15)
    body = co.compress(text) + co.flush()
    xlen = len(before) + 6 + len(after)
    bsize = 12 + xlen + len(body) + 8 if bsize is None else bsize
    extra = before + b"BC" + struct.pack("<HH", 2, bsize - 1) + after
    return member(body, text, extra=extra)


def bgzf_files():
    rng = random.Random(9)
    texts = [bed_text(rng, n) for n in (200, 1, 0, 900, 50)]
    sub_a, sub_b = b"XY" + struct.pack("<H", 3) + b"abc", b"ZZ" + struct.pack("<H", 0)
    files = {
        "bc_after_other_subfields": [bgzf_member(t, before=sub_a + sub_b) for t in texts],
        "subfields_before_and_after_bc": [bgzf_member(t, before=sub_a, after=sub_b + sub_a) for t in texts],
        "bc_first_then_subfields": [bgzf_member(t, after=sub_b) for t in texts],
    }
    out = {k: ([len(m) for m in ms], b"".join(ms), b"".join(texts)) for k, ms in files.items()}
    # a BSIZE that points past the end of the file: the splitter takes the rest of the file as one member, which the device
    # then rejects (two members in one unit)
    ms = [bgzf_member(texts[0]), bgzf_member(texts[1]), bgzf_member(texts[4], bsize=65536), bgzf_member(texts[3])]
    assert sum(len(m) for m in ms[2:]) < 65536
    out["bsize_past_end"] = ([len(ms[0]), len(ms[1]), len(ms[2]) + len(ms[3])], b"".join(ms), None)
    # BGZF members, then a plain gzip member (no FEXTRA): the tail is one member
    ms = [bgzf_member(t) for t in texts] + [gzip.compress(b"plain tail\n" * 50, mtime=0)]
    out["plain_gzip_tail"] = ([len(m) for m in ms], b"".join(ms), b"".join(texts) + b"plain tail\n" * 50)
    return out


# ---- host checks: no GPU ----------------------------------------------------------------------------------------------------
def test_writer_streams_match_zlib():
    """Every valid stream the writer makes decodes with zlib to the text the writer meant."""
    cases = valid_cases()
    assert len(cases) > 500
    for name, (m, text) in cases.items():
        assert zlib_inflate(m) == text, name


def test_writer_invalid_streams_are_rejected_by_zlib():
    for name, (m, _) in invalid_cases().items():
        assert zlib_inflate(m) is None, name


def test_writer_codes_reach_the_lengths_they_are_meant_to():
    """The random deep trees really use codes of 10 bits (the last first-level length) and 11..15 bits."""
    seen_ll, seen_d = set(), set()
    for seed in range(8):
        r = random.Random(100 + seed)
        toks = random_tokens(r, 3000, r.sample(range(256), 40), dist_codes=r.sample(range(30), 12), size=0)
        u_ll, u_d = used_symbols(toks)
        ll, d = deep(u_ll, r), deep(u_d, r)
        seen_ll |= {ll[s] for s in u_ll}
        seen_d |= {d[s] for s in u_d}
    assert set(range(10, 16)) <= seen_ll and {9, 10, 11} <= seen_d  # longer distance codes: ll_1_to_15_bits_d_1_to_15_bits


def test_gzip_members_splits_bgzf_extra_fields():
    from gtars_b200 import ffi
    for name, (sizes, gz, _) in bgzf_files().items():
        assert list(ffi.gzip_members(gz)) == [0, *np.cumsum(sizes)], name


# ---- on the device ------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def ctx():
    from gtars_b200 import ffi
    c = ffi.Context(0)
    yield c
    c.close()


def offsets(sizes, base=0):
    return np.concatenate([[base], base + np.cumsum(sizes, dtype=np.uint64)]).astype(np.uint64)


def gunzip_checked(ctx, members, texts, base=b""):
    """gtgpu_gunzip of the members back to back (behind `base` junk bytes) == zlib, text and member offsets."""
    from gtars_b200 import ffi
    gz = base + b"".join(members)
    got, off = ffi.gunzip(ctx, gz, offsets([len(m) for m in members], len(base)))
    assert list(off) == list(offsets([len(t) for t in texts]))
    for k, t in enumerate(texts):
        assert got[int(off[k]):int(off[k + 1])] == t, k
    return got


@pytest.mark.gpu
@pytest.mark.parametrize("group", ["tree", "match", "literal_run", "stored", "ring", "zlib", "size"])
def test_valid_streams_match_zlib(ctx, group):
    cases = globals()[f"{group}_cases"]()
    for name, (m, text) in cases.items():
        assert gunzip_checked(ctx, [m], [text]) == text, name
    ms, ts = zip(*cases.values())
    gunzip_checked(ctx, list(ms), list(ts))


@pytest.mark.gpu
def test_all_valid_streams_in_one_call_at_odd_offsets(ctx):
    """Every case as a member of one call, behind 5 junk bytes: members at unaligned offsets, a nonzero base, and the
    last trailer ending the buffer exactly."""
    ms, ts = zip(*valid_cases().values())
    gunzip_checked(ctx, list(ms), list(ts), base=b"\x1f\x8b\x08\0\0")


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(invalid_cases()))
def test_invalid_stream_reports_its_reason(ctx, name):
    from gtars_b200 import ffi
    bad, reason = invalid_cases()[name]
    assert zlib_inflate(bad) is None
    good_a, ta = Deflate().dynamic(list(b"a good member before\n") + [(12, 5)], True).member()
    good_b, tb = member(b"\x03\x00", b""), b""
    pat = (lambda k: f"member {k} {re.escape(reason)}$") if reason == SHORT else (lambda k: f"member {k}: {re.escape(reason)}$")
    with pytest.raises(ffi.GtarsGpuError, match=pat(0)):
        ffi.gunzip(ctx, bad, offsets([len(bad)]))
    with pytest.raises(ffi.GtarsGpuError, match=pat(1)):
        ffi.gunzip(ctx, good_a + bad + good_b, offsets([len(good_a), len(bad), len(good_b)]))
    gunzip_checked(ctx, [good_a, good_b], [ta, tb])


@pytest.mark.gpu
def test_more_members_than_the_resident_grid(ctx):
    """About 4x as many members as the grid has warps at the highest occupancy an SM allows (64 warps): the grid-stride
    loop runs and every warp's shared tables and ring are reused for members of every kind, tiny, empty and large."""
    import torch
    n = 4 * torch.cuda.get_device_properties(0).multi_processor_count * 64
    rng = random.Random(10)
    pool = bed_text(rng, 8000)
    big = [gzip.compress(pool[k * 1000:], compresslevel=lv, mtime=0) for k, lv in enumerate((0, 1, 6, 9))]
    ms, ts = [], []
    for k in range(n):
        if k % 5000 == 17:
            j = (k // 5000) % 4
            ms.append(big[j])
            ts.append(pool[j * 1000:])
            continue
        t = b"" if k % 3 == 0 else pool[k % 7919:k % 7919 + k % 61]
        ms.append(gzip.compress(t, compresslevel=k % 10, mtime=0))
        ts.append(t)
    gunzip_checked(ctx, ms, ts, base=b"xyz")


@pytest.mark.gpu
def test_one_member_of_32_mib(ctx):
    """The one-member universe shape: 32 MiB of BED-like text in a single member, decoded by one warp (seconds)."""
    from gtars_b200 import synth
    c, s, e, b = synth.make_fragment_arrays((32 << 20) // synth.FRAGMENT_LINE + 1, 11, 5000)
    text = synth.fragment_text(c, s, e, b).tobytes()
    m = gzip.compress(text, compresslevel=6, mtime=0)
    assert len(text) >= 32 << 20 and zlib_inflate(m) == text
    assert gunzip_checked(ctx, [m], [text]) == text


@pytest.mark.gpu
def test_bgzf_extra_fields_decode(ctx):
    from gtars_b200 import ffi
    for name, (_, gz, text) in bgzf_files().items():
        if text is None:
            with pytest.raises(ffi.GtarsGpuError, match=f"member 2: {TRAILING}$"):
                ffi.gunzip(ctx, gz)
            continue
        got, off = ffi.gunzip(ctx, gz)
        assert got == text and int(off[-1]) == len(text), name


def three_block_member(text, seed):
    """text as one member of a stored, a fixed and a dynamic block whose used codes reach 15 bits."""
    a = min(len(text) // 5, 65535)  # one stored block holds at most 65535 bytes
    b = 2 * a
    r = random.Random(seed)
    rest = list(text[b:])
    u = set(rest) | {256}
    while True:
        ll = deep(u, r)
        if max(ll[s] for s in u) == 15:
            break
    d = Deflate().stored(text[:a]).fixed(list(text[a:b])).dynamic(rest, True, ll=ll, d={})
    m, t = d.member()
    assert t == text and zlib_inflate(m) == text
    return m


@pytest.mark.gpu
def test_member_with_every_block_kind_through_the_parsers(ctx):
    """tokenize_bed_gz and score_matrix_gz of a member with stored, fixed and 15-bit dynamic blocks == their text forms."""
    from gtars_b200 import ffi, synth
    u = synth.make_universe(30_000)
    offs = u["chrom_offsets"].numpy().astype(np.uint64)
    s, e, v = (u[k].numpy().view(np.uint32) for k in ("g_start", "g_end", "g_val"))
    ix = ffi.Index(ctx, ffi.KIND_BITS, offs, s, e, v)
    try:
        names = list(synth.CHROM_NAMES)
        q = synth.make_query_files(u, 1, 20_000, unknown_frac_ppm=300)
        qc, qs, qe = (q[k].numpy() for k in ("chr", "start", "end"))
        name_arr = np.array(names + ["chrUn"])
        bed = ("\n".join(map("\t".join, zip(name_arr[qc], qs.astype(str), qe.astype(str)))) + "\n").encode()
        m = three_block_member(bed, 12)
        want = ix.tokenize_bed(bed, names, int(u["unk_id"]))
        assert len(want) > 0
        assert np.array_equal(ix.tokenize_bed_gz(m, names, int(u["unk_id"]), member_offsets=offsets([len(m)])), want)
        c, fs, fe, b = synth.make_fragment_arrays(20_000, 13, 300)
        frag = synth.fragment_text(c, fs, fe, b).tobytes()
        fm = three_block_member(frag, 14)
        for mode in (ffi.SCORE_ATAC, ffi.SCORE_CHIP):
            want = ix.score_matrix_text(frag, names, mode, int(u["n"]))
            got = ix.score_matrix_text(fm, names, mode, int(u["n"]), gz_member_offsets=offsets([len(fm)]))
            assert np.array_equal(got, want), mode
    finally:
        ix.close()
