"""The IGD count kernel (igd_count_kernel<BINARY, M1> in igd.cu) against two references, at its instantiations and edges.

The kernel keeps, per chromosome, one start-sorted pool of every database record plus the running maximum of their ends
(pmax); a query's candidates are the run [first i with pmax > s, #starts < e), found by two warp-cooperative lower bounds
(lb_warp) from LUT bins of 2^shift bp, and tested 128 candidates per round.  count_region_hits counts a (query, file) pair
once through psame (the largest end of an earlier same-file record at least m long).  Each case here aims at one of these
parts: kernel instantiations and grid shapes, candidate runs at round edges, long runs of candidates that do not hit,
lower-bound ranges of every size, int32 semantics of igd.rs, psame across rounds and m values, wide build shapes, and the
device entry point's accumulation.

References:
  oracle.Igd   replays the reference's 16 384-bp tile walk (igd.rs:504-540, 753-847), independent of the pooled design;
  ref_counts   the plain definition in numpy, below.  test_ref_counts_matches_oracle (no GPU needed) shows that the two
               agree on every case of this file before either is used against the kernel.

Run-time knobs of the count (read on every call): GTGPU_IGD_NO_M1=1 runs the general kernel at min_overlap = 1, and
GTGPU_IGD_CTAS=1 shrinks the grid to one block per SM, so each warp strides through many queries (the next-query prefetch).
"""
import contextlib
import os
import types
import zlib

import numpy as np
import pytest

gpu = pytest.mark.gpu

I32_MAX = 2**31 - 1
TILE = 16_384          # the reference's tile (igd.rs:79-81)
ROUND = 128            # candidates per round of igd_count_kernel: 4 loads per lane of a warp
WARPS_PER_BLOCK = 8    # igd_count_kernel runs 256-thread blocks, one warp per query

KERNELS = (("m1", {"GTGPU_IGD_NO_M1": None}), ("general", {"GTGPU_IGD_NO_M1": "1"}))
GRIDS = (("default grid", {"GTGPU_IGD_CTAS": None}), ("one block per SM", {"GTGPU_IGD_CTAS": "1"}))


def rng_for(name):
    return np.random.default_rng(zlib.crc32(name.encode()))


def offsets(sizes):
    return np.concatenate([[0], np.cumsum(np.asarray(sizes, np.int64))]).astype(np.uint64)


def u32(a):
    return np.asarray(np.asarray(a, np.int64) & 0xFFFFFFFF, np.uint32)


def make_case(file_records, n_chroms, set_queries, ms):
    """file_records: per file a list / array of (chr, start, end); set_queries: per set a list of (chr, start, end).  Coordinates
    are taken modulo 2^32, as the uint32 arrays of the C ABI carry them."""
    def flat(groups):
        groups = [np.asarray(g, np.int64).reshape(-1, 3) for g in groups]
        a = np.concatenate(groups) if groups else np.zeros((0, 3), np.int64)
        return offsets([len(g) for g in groups]), u32(a[:, 0]), u32(a[:, 1]), u32(a[:, 2])
    fo, chr_, start, end = flat(file_records)
    so, qc, qs, qe = flat(set_queries)
    return types.SimpleNamespace(fo=fo, n_chroms=n_chroms, chr=chr_, start=start, end=end, so=so, qc=qc, qs=qs, qe=qe, ms=tuple(ms))


# ---- the plain definition ------------------------------------------------------------------------------------------------
def kept_records(case):
    """(chr, start, end, file) of the records Igd::from_named_region_sets keeps: start < end as u32 (igd.rs:285-301), then
    Igd::add's 0 <= start < end as i32 (igd.rs:109-116); coordinates as int64."""
    n_files = len(case.fo) - 1
    rf = np.repeat(np.arange(n_files, dtype=np.int64), np.diff(case.fo.astype(np.int64)))
    rs, re = case.start.view(np.int32).astype(np.int64), case.end.view(np.int32).astype(np.int64)
    keep = (case.start < case.end) & (rs >= 0) & (re >= 0)
    return case.chr[keep], rs[keep], re[keep], rf[keep]


def ref_counts(case, m, binary):
    """uint64 [n_sets, n_files]: count_set_overlaps (binary=False: every hit counts) or count_region_hits (binary=True: a
    (query, file) pair counts once).  A query (chr, s, e) cast to int32 counts nothing when s >= e or e <= 0, else s clamps
    to 0 (igd.rs:514-522); a kept record r of the same chromosome hits iff min(r.end, e) - max(r.start, s) >= m."""
    rc, rs, re, rf = kept_records(case)
    n_files, n_sets = len(case.fo) - 1, len(case.so) - 1
    qset = np.repeat(np.arange(n_sets, dtype=np.int64), np.diff(case.so.astype(np.int64)))
    qs, qe = case.qs.view(np.int32).astype(np.int64), case.qe.view(np.int32).astype(np.int64)
    live = np.flatnonzero((qs < qe) & (qe > 0))
    qs = np.maximum(qs, 0)
    order = np.argsort(rc, kind="stable")
    rc_sorted = rc[order]
    cells = []
    for c in np.unique(case.qc[live]):
        lo, hi = np.searchsorted(rc_sorted, c, "left"), np.searchsorted(rc_sorted, c, "right")
        if lo == hi:
            continue
        r = order[lo:hi]
        r_s, r_e, r_f = rs[r], re[r], rf[r]
        qq = live[case.qc[live] == c]
        step = max(1, (1 << 22) // len(r))
        for i in range(0, len(qq), step):
            q = qq[i:i + step]
            ov = np.minimum(r_e[None, :], qe[q][:, None]) - np.maximum(r_s[None, :], qs[q][:, None])
            qi, ri = np.nonzero(ov >= m)
            pair = q[qi] * n_files + r_f[ri]
            if binary:
                pair = np.unique(pair)
            cells.append(qset[pair // n_files] * n_files + pair % n_files)
    flat = np.concatenate(cells) if cells else np.zeros(0, np.int64)
    return np.bincount(flat, minlength=n_sets * n_files).astype(np.uint64).reshape(n_sets, n_files)


def expected_shift(case):
    """The LUT shift igd_build_dev chooses: the least shift whose bins (last running max >> shift, plus 2, per populated
    chromosome) fit a budget of max(kept records, 4 096), at most 8 Mi, capped at 31."""
    rc, _, re, _ = kept_records(case)
    last = np.zeros(case.n_chroms, np.int64)
    np.maximum.at(last, rc.astype(np.int64), re)
    populated = np.bincount(rc, minlength=case.n_chroms) > 0
    budget = min(max(len(rc), 4096), 8 << 20)
    shift = 0
    while shift < 31 and int(((last[populated] >> shift) + 2).sum()) > budget:
        shift += 1
    return shift


# ---- cases -----------------------------------------------------------------------------------------------------------------
def case_mixed():
    """64 files (empty ones among them, the last one too), 5 chromosomes with chromosome 3 empty, dropped records (reversed,
    empty, negative as int32), records spanning up to 120 tiles; query sets of 0, 1 and many queries, with empty, reversed,
    negative-start and unknown-chromosome queries."""
    rng = rng_for("mixed")
    n_chroms, n_files = 5, 64
    sizes = rng.integers(0, 300, n_files)
    sizes[[0, 7, 31, 63]] = 0
    files = []
    for f in range(n_files):
        n = int(sizes[f])
        c = rng.choice([0, 1, 2, 4], n)
        s = rng.integers(0, 3_000_000, n)
        w = rng.integers(1, 60, n)
        kind = rng.random(n)
        w = np.where(kind < 0.3, rng.integers(60, 40_000, n), w)
        w = np.where(kind < 0.03, rng.integers(200_000, 2_000_000, n), w)
        e = s + w
        e = np.where((kind > 0.95) & (kind < 0.97), s, e)                    # empty
        e = np.where((kind > 0.97) & (kind < 0.98), s - 5, e)                # reversed
        s = np.where(kind > 0.99, s + 2**31, s)                              # negative start as int32: dropped
        e = np.where(kind > 0.99, s + 100, e)
        files.append(np.stack([c, s, e], 1))
    sets = []
    for n in (0, 1, 900, 0, 1500, 37, 1):
        c = rng.choice([0, 1, 2, 3, 4, 5, 0xFFFFFFFF], n, p=[0.25, 0.2, 0.2, 0.05, 0.2, 0.05, 0.05])
        s = rng.integers(0, 3_100_000, n)
        e = s + rng.integers(1, 60_000, n)
        kind = rng.random(n)
        e = np.where(kind < 0.04, s, e)                                      # empty
        e = np.where((kind > 0.04) & (kind < 0.07), s - 3, e)                # reversed
        s = np.where(kind > 0.96, 2**32 - rng.integers(1, 5_000, n), s)      # negative start: clamps to 0
        sets.append(np.stack([c, s, e], 1))
    return make_case(files, n_chroms, sets, ms=(1, 2, 100))


def rounds_layout(layout):
    """Records [2i, 2i + 2), i < 10 000, on chromosome 0: in files of 64 consecutive records (blocks) or record i in file
    i mod 7 (interleaved).  Returns (file of record i, n_files)."""
    i = np.arange(10_000)
    return (i // 64, 157) if layout == "blocks" else (i % 7, 7)


ROUND_KS = (1, 2, 31, 32, 33, 95, 96, 97, 127, 128, 129, 255, 256, 257, 4096, 4097)
ROUND_PHASES = (0, 1, 31, 96, 127)
ROUND_T = (3, 17, 30)


def case_rounds(layout):
    """Query [2a, 2a + 2k) has exactly the k candidates i in [a, a + k) (pmax > 2a, start < 2a + 2k), all hitting by 2 bp:
    k around multiples of the round, a mod 128 at every phase.  One set per query."""
    file_of, n_files = rounds_layout(layout)
    i = np.arange(len(file_of))
    files = [np.stack([np.zeros(int((file_of == f).sum())), 2 * i[file_of == f], 2 * i[file_of == f] + 2], 1) for f in range(n_files)]
    sets = [[(0, 2 * a, 2 * (a + k))] for a, k in round_queries()]
    return make_case(files, 1, sets, ms=(1, 2, 3))


def round_queries():
    return [(ROUND * t + r, k) for k in ROUND_KS for r in ROUND_PHASES for t in ROUND_T]


def case_nonhit():
    """Per chromosome one record of file 0 covers everything, so pmax is flat and every query's run starts at the first
    record: thousands of candidates, most of which do not hit.  Short records of widths 1..7 (m - 1, m, m + 1 of every m
    tested) in 40 files; queries that touch records (s = a record's end, e = a record's start), queries narrower than m, and
    random ones."""
    rng = rng_for("nonhit")
    n_chroms, n_files = 3, 41
    spans = (1_000_000, 200_000, 3_000_000)
    recs = [[] for _ in range(n_files)]
    for c, span in enumerate(spans):
        recs[0].append((c, 0, span))
        n = 5000
        s = rng.integers(0, span - 10, n)
        w = rng.integers(1, 8, n)
        w = np.where(rng.random(n) < 0.1, rng.integers(8, 5000, n), w)
        f = rng.integers(1, n_files, n)
        for a, b, ff in zip(s, s + w, f):
            recs[ff].append((c, int(a), int(b)))
    all_recs = np.array([r for rr in recs[1:] for r in rr], np.int64)
    sets = []
    for _ in range(4):
        pick = all_recs[rng.integers(0, len(all_recs), 300)]
        wq = rng.integers(1, 9, 300)
        touch_after = np.stack([pick[:, 0], pick[:, 2], pick[:, 2] + wq], 1)      # starts where a record ends
        touch_before = np.stack([pick[:, 0], pick[:, 1] - wq, pick[:, 1]], 1)     # ends where a record starts
        inside = np.stack([pick[:, 0], pick[:, 1], pick[:, 1] + rng.integers(1, 4, 300)], 1)  # narrower than most m
        c = rng.integers(0, n_chroms, 200)
        s = rng.integers(0, 3_000_000, 200)
        rand = np.stack([c, s, s + rng.integers(1, 20_000, 200)], 1)
        sets.append(np.concatenate([touch_after, touch_before, inside, rand]))
    return make_case([np.array(r) for r in recs], n_chroms, sets, ms=(1, 2, 5, 6))


def case_lb_cluster():
    """(i) 20 000 records in the first 4 kb of chromosome 0 and one record ending at 2^31 - 1 on the same chromosome: the shift
    is at least 15 and the first start bin and the first pmax bin hold the whole cluster."""
    rng = rng_for("lb_cluster")
    n_files = 40
    sizes = rng.multinomial(20_000, np.ones(n_files) / n_files)
    files = []
    for f in range(n_files):
        s = rng.integers(0, 4096, sizes[f])
        files.append(np.stack([np.zeros_like(s), s, s + rng.integers(1, 300, sizes[f])], 1))
    files[-1] = np.concatenate([files[-1], [[0, I32_MAX - 1000, I32_MAX]]])
    files[3] = np.concatenate([files[3], [[1, 10, 5000], [1, 2**30, 2**30 + 7]]])
    s = rng.integers(0, 4400, 1500)
    rand = np.stack([np.zeros_like(s), s, s + rng.integers(1, 400, 1500)], 1)
    edges = []
    for b in (131_072, 2**31 - 131_072):
        for d in (-1, 0, 1):
            edges += [(0, 0, b + d), (0, b + d - 1, b + d + 5), (0, b + d - 1, I32_MAX)]
    edges += [(0, I32_MAX - 1, I32_MAX), (1, 0, 2**30 + 1), (0, 2000, 2001), (0, 4095, 4096)]
    return make_case(files, 2, [rand[:700], edges, rand[700:]], ms=(1, 2, 50))


SHARED_COUNTS = (2000, 1025, 64, 33, 32, 31, 1)


def case_lb_shared():
    """(ii) 2 000 files sharing 50 regions: region j is held by the first SHARED_COUNTS[j % 7] files, so its start bin holds
    2 000, 1 025, 64, 33, 32, 31 or 1 equal starts, and its end a pmax plateau of as many records.  Queries put e on the
    last base of a start bin and s + 1 on pmax bin edges (+-1)."""
    rng = rng_for("lb_shared")
    n_files = 2000
    starts = 20_000 * np.arange(50) + 5_001 + rng.integers(0, 30, 50)
    widths = 100 + 37 * np.arange(50)
    files = [[] for _ in range(n_files)]
    for j in range(50):
        for f in range(SHARED_COUNTS[j % 7]):
            files[f].append((0, int(starts[j]), int(starts[j] + widths[j])))
    shift = 6  # asserted in the test
    q = []
    for j in range(50):
        s0, e0 = int(starts[j]), int(starts[j] + widths[j])
        bin_end = ((s0 >> shift) + 1) << shift
        for e in (bin_end - 1, bin_end, bin_end + 1, s0 + 1, e0):
            q.append((0, s0, e))
            q.append((0, s0 - 3, e))
        for b in ((e0 >> shift) << shift, ((e0 >> shift) + 1) << shift):
            for d in (-2, -1, 0, 1):
                q.append((0, b + d - 1, b + d + 40))    # s + 1 = b + d
    q = np.array(q, np.int64)
    s = rng.integers(0, 1_000_000, 400)
    rand = np.stack([np.zeros_like(s), s, s + rng.integers(1, 3000, 400)], 1)
    return make_case([np.array(r, np.int64) for r in files], 1, [q[::2], q[1::2], rand], ms=(1, 2, 70))


def case_lb_plateau():
    """(iii) Rising ends for 3 000 records, then one record to 2 000 000 and 5 000 short records after it: the running maximum
    is flat over a bin of more than 5 000 records.  A few records just before the wide one end inside that bin."""
    rng = rng_for("lb_plateau")
    n_files = 23
    rec = [(0, 10 * i, 10 * i + 15) for i in range(3000)]
    rec += [(0, 29_990 + j, 1_999_800 + 9 * j) for j in range(10)]
    rec += [(0, 30_000, 2_000_000)]
    s = np.sort(rng.integers(30_001, 1_999_000, 5000))
    rec += [(0, int(a), int(a + w)) for a, w in zip(s, rng.integers(1, 500, 5000))]
    rec = np.array(rec, np.int64)
    f = rng.integers(0, n_files, len(rec))
    files = [rec[f == k] for k in range(n_files)]
    q = []
    for b in range(1_999_000 >> 8, (2_000_100 >> 8) + 1):
        for d in (-1, 0, 1):
            q.append((0, (b << 8) + d - 1, (b << 8) + d + 30))
    for b in range(0, 30_100 >> 8):
        q.append((0, (b << 8) - 1, (b << 8) + 3))
        q.append((0, (b << 8), (b << 8) + 1))
    s = rng.integers(0, 2_001_000, 600)
    rand = np.stack([np.zeros_like(s), s, s + rng.integers(1, 3000, 600)], 1)
    return make_case(files, 1, [np.array(q, np.int64), rand], ms=(1, 2, 31))


DENSE_COUNTS = (31, 32, 33, 64, 1025)


def case_lb_dense():
    """(iv) A dense chromosome with shift 0: every bp is a bin.  Groups of 31, 32, 33, 64 and 1 025 records share one start,
    with ends spread over the next 3 kb; a background of [i, i + 3) records keeps the shift at 0."""
    rng = rng_for("lb_dense")
    n_files = 9
    rec = [(0, i, i + 3) for i in range(0, 5000)]
    for g, cnt in enumerate(DENSE_COUNTS):
        p = 400 + 700 * g
        rec += [(0, p, p + int(w)) for w in rng.integers(1, 1200, cnt)]
    rec = np.array(rec, np.int64)
    f = rng.integers(0, n_files, len(rec))
    files = [rec[f == k] for k in range(n_files)]
    q = []
    for g in range(len(DENSE_COUNTS)):
        p = 400 + 700 * g
        for d in (-1, 0, 1, 2):
            q += [(0, p + d - 1, p + d), (0, p - 5, p + d), (0, p + d, p + d + 700)]
    s = rng.integers(0, 5100, 500)
    rand = np.stack([np.zeros_like(s), s, s + rng.integers(1, 600, 500)], 1)
    return make_case(files, 1, [np.array(q, np.int64), rand], ms=(1, 2, 300))


INT32_RECORDS = (
    # file 0: two records ending at 2^31 - 1 (the largest end kept), widths 99 and 49
    [(0, 2**31 - 100, 2**31 - 1), (0, 2**31 - 50, 2**31 - 1)],
    # file 1: [2^31 - 1, 2^31) and [1000, 2^31) end past int32 (dropped), [2^31, 2^31 + 10) starts negative (dropped),
    # [5, 5) and [7, 3) are not regions (dropped); [0, 1) is kept
    [(0, 2**31 - 1, 2**31), (0, 1000, 2**31), (0, 2**31, 2**31 + 10), (0, 5, 5), (0, 7, 3), (0, 0, 1),
     (1, 2**32 - 6, 2**32 - 1), (1, 2**31 - 2, 2**31 + 1)],
    # file 2: records on and across the 16 384-bp tile boundaries, and one record over the whole int32 range
    [(0, TILE - 1, TILE + 1), (0, TILE, TILE + 1), (0, 2 * TILE - 1, 2 * TILE), (0, 3 * TILE, 5 * TILE + 7), (0, 0, I32_MAX),
     (1, TILE - 2, TILE), (1, 10, 20)],
    # file 3: empty
    [],
    # file 4: records of 1, 2, 49, 50 and 51 bp around 2^30
    [(1, 2**30, 2**30 + w) for w in (1, 2, 49, 50, 51)],
)
INT32_KEPT = 2 + 1 + 7 + 5


def int32_queries(n_chroms):
    q = [(0, 0xFFFFFFF0, 100), (0, 100, 0x80000000), (0, 0x7FFFFFFE, 0x7FFFFFFF), (0, 0, 0x7FFFFFFF), (1, 0, 0x7FFFFFFF),
         (0, 0xFFFFFFF0, 0xFFFFFFFF), (0, 0x80000000, 0x80000001), (0, 0x7FFFFFFF, 0x80000000), (0, 2**31 - 60, 2**31 - 10),
         (1, 0xFFFFFFFF, 2**30 + 1), (1, 2**30 - 1, 2**30 + 50), (1, 2**30, 2**30 + 51), (1, 2**30 + 1, 2**30 + 2)]
    for k in (1, 2, 3, 5):
        for d in (-1, 0, 1):
            b = k * TILE + d
            q += [(0, b - 1, b), (0, b, b + 1), (0, b - 1, b + 1), (1, b - 2, b), (0, b, 7 * TILE)]
    for c in (n_chroms, n_chroms + 5, 0xFFFFFFFF):
        q += [(c, 0, 100), (c, 0, 0x7FFFFFFF)]
    return q


def case_int32(extra_chroms=0):
    """int32 semantics of Igd::add and count_overlaps.  extra_chroms > 0 adds that many chromosomes with one record ending at
    2^31 - 1 each (in file 3), which drives the LUT shift up to 25 (the oracle keeps 131 072 tiles per such chromosome, so
    their number stays small)."""
    files = [list(f) for f in INT32_RECORDS]
    n_chroms = 3 + extra_chroms
    files[3] = [(3 + c, 2**31 - 2 - c, I32_MAX) for c in range(extra_chroms)]
    q = int32_queries(n_chroms)
    return make_case(files, n_chroms, [q[::2], [], q[1::2]], ms=(1, 2, 50, 100))


def case_psame():
    """A query [S, S + 1000) whose candidates start with a record of file 0 covering everything, then more than a round of
    records of files 1..7 that end at or before S, then in rounds 2 and 3 the hits of files 1..6: first a record of exactly
    f bp inside the query (file f), then two later records of the same file that hit by 10 bp.  File 7 has one record
    reaching into the query from round 1 and 60 short ones after it."""
    rng = rng_for("psame")
    n_files = 8
    S = 100_000
    files = [[] for _ in range(n_files)]
    files[0].append((0, 0, 10_000_000))
    # round 1: 200 non-hits of files 1..7 that start before the query and end at or before S
    for j in range(200):
        f = 1 + j % 7
        a = S - 5000 + 20 * j
        files[f].append((0, a, min(a + 15, S)))
    # rounds 2 and 3: the first hit of file f is f bp long, then two 10-bp hits of the same file
    for j, f in enumerate(range(1, 7)):
        files[f].append((0, S + 100 + j, S + 100 + j + f))
    for j, f in enumerate(range(1, 7)):
        files[f].append((0, S + 300 + j, S + 310 + j))
        files[f].append((0, S + 500 + j, S + 510 + j))
    # file 7: a long record early that reaches into the query, so its psame is set from round 1
    files[7].append((0, S - 4000, S + 50))
    for j in range(60):
        files[7].append((0, S + 600 + j, S + 605 + j))
    s = rng.integers(S - 6000, S + 1200, 300)
    rand = np.stack([np.zeros_like(s), s, s + rng.integers(1, 1500, 300)], 1)
    fixed = [(0, S + d, S + 1000) for d in (-1, 0, 1, 50, 99, 100, 101, 105, 106, 300)]
    return make_case([np.array(r, np.int64) for r in files], 1, [fixed, rand], ms=(2, 5, 2, 1, 5, 3))


WIDE = 70_001


def case_wide_files():
    """70 001 files of one or two records over 3 chromosomes: the file radix pass of the psame build takes 17 bits."""
    rng = rng_for("wide_files")
    sizes = rng.integers(1, 3, WIDE)
    n = int(sizes.sum())
    c = rng.integers(0, 3, n)
    s = rng.integers(0, 5_000_000, n)
    rec = np.stack([c, s, s + rng.integers(1, 20_000, n)], 1)
    fo = offsets(sizes).astype(np.int64)
    files = [rec[fo[f]:fo[f + 1]] for f in range(WIDE)]
    qs = rng.integers(0, 5_000_000, 300)
    q = np.stack([rng.integers(0, 4, 300), qs, qs + rng.integers(1, 100_000, 300)], 1)
    return make_case(files, 3, [q[:100], q[100:101], q[101:]], ms=(1, 2))


def case_wide_chroms():
    """70 001 chromosome ids of which 300 scattered ones (the first and the last among them) hold records: the chromosome radix
    passes take 17 bits, and populated chromosomes have empty ones between them."""
    rng = rng_for("wide_chroms")
    populated = np.unique(np.concatenate([[0, WIDE - 1], rng.choice(WIDE, 298, replace=False)]))
    n_files = 37
    n = 12_000
    c = rng.choice(populated, n)
    s = rng.integers(0, 1_000_000, n)
    rec = np.stack([c, s, s + rng.integers(1, 30_000, n)], 1)
    f = rng.integers(0, n_files, n)
    files = [rec[f == k] for k in range(n_files)]
    nq = 1500
    qc = np.where(rng.random(nq) < 0.8, rng.choice(populated, nq), rng.integers(0, WIDE + 3, nq))
    qs = rng.integers(0, 1_000_000, nq)
    q = np.stack([qc, qs, qs + rng.integers(1, 50_000, nq)], 1)
    return make_case(files, WIDE, [q[:700], q[700:]], ms=(1, 3))


CASES = {
    "mixed": case_mixed,
    "rounds_blocks": lambda: case_rounds("blocks"),
    "rounds_interleaved": lambda: case_rounds("interleaved"),
    "nonhit": case_nonhit,
    "lb_cluster": case_lb_cluster,
    "lb_shared": case_lb_shared,
    "lb_plateau": case_lb_plateau,
    "lb_dense": case_lb_dense,
    "int32": case_int32,
    "int32_high_shift": lambda: case_int32(40),
    "psame": case_psame,
    "wide_files": case_wide_files,
    "wide_chroms": case_wide_chroms,
}


# ---- harness -----------------------------------------------------------------------------------------------------------------
def oracle_counts(o, case, m, binary):
    from oracle import oracle as orc
    fn = o.count_region_hits if binary else o.count_set_overlaps
    return fn(case.so, case.qc, case.qs, case.qe, m, threads=orc.max_threads())


def make_oracle(case):
    from oracle import oracle as orc
    return orc.Igd(case.fo, case.chr, case.start, case.end)


def assert_counts(got, want, label):
    assert got.shape == want.shape, f"{label}: shape {got.shape} != {want.shape}"
    bad = np.argwhere(got != want)
    assert len(bad) == 0, (f"{label}: {len(bad)} of {want.size} cells differ, e.g. (set, file, got, want) "
                           + ", ".join(f"({s}, {f}, {got[s, f]}, {want[s, f]})" for s, f in bad[:6]))


@contextlib.contextmanager
def knobs(settings):
    """Set (value) or unset (None) environment variables for the duration; the library reads them on every count."""
    old = {k: os.environ.get(k) for k in settings}
    try:
        for k, v in settings.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v
        yield
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


def device_counts(g, case, m, binary):
    fn = g.count_region_hits if binary else g.count_set_overlaps
    return fn(case.so, case.qc, case.qs, case.qe, m)


def check_variants(g, case, name, ms=None, o=None, with_ref=True, grids=GRIDS):
    """Both semantics at every m of the case, every kernel that serves that m (m = 1: M1 and the general kernel) and every grid
    shape, against the oracle (and ref_counts); the two kernels at m = 1 against each other."""
    o = o if o is not None else make_oracle(case)
    for m in ms or case.ms:
        for binary in (False, True):
            sem = "count_region_hits" if binary else "count_set_overlaps"
            want = oracle_counts(o, case, m, binary)
            if with_ref:
                assert_counts(ref_counts(case, m, binary), want, f"{name}: ref_counts vs oracle, m={m} {sem}")
            first = None
            for kname, kenv in (KERNELS if m == 1 else KERNELS[1:]):
                for gname, genv in grids:
                    with knobs({**kenv, **genv}):
                        got = device_counts(g, case, m, binary)
                    assert_counts(got, want, f"{name}: m={m} {sem}, {kname} kernel, {gname}")
                    if first is None:
                        first = got
                    assert np.array_equal(got, first), f"{name}: m={m} {sem}: {kname} kernel, {gname} disagrees with the first variant"


@pytest.fixture(scope="module")
def ctx():
    from gtars_b200 import ffi
    c = ffi.Context(0)
    yield c
    c.close()


def build(ctx, case):
    from gtars_b200 import ffi
    return ffi.Igd(ctx, case.fo, case.n_chroms, case.chr, case.start, case.end)


# ---- the two references agree (no GPU) ---------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", sorted(CASES))
def test_ref_counts_matches_oracle(name):
    """ref_counts and the oracle's tile walk agree on every case of this file, at every m the case uses, both semantics."""
    case = CASES[name]()
    o = make_oracle(case)
    for m in sorted(set(case.ms)):
        for binary in (False, True):
            assert_counts(ref_counts(case, m, binary), oracle_counts(o, case, m, binary),
                          f"{name}: m={m} {'count_region_hits' if binary else 'count_set_overlaps'}")


def test_round_cases_closed_form():
    """The round cases' queries count exactly k pairs (records [2i, 2i + 2) with i in [a, a + k)) at m = 1 and 2, none at m = 3."""
    for layout in ("blocks", "interleaved"):
        case = case_rounds(layout)
        file_of, n_files = rounds_layout(layout)
        want = np.stack([np.bincount(file_of[a:a + k], minlength=n_files) for a, k in round_queries()]).astype(np.uint64)
        for m in (1, 2):
            assert_counts(ref_counts(case, m, False), want, f"rounds {layout}: m={m} pairs")
            assert_counts(ref_counts(case, m, True), (want > 0).astype(np.uint64), f"rounds {layout}: m={m} hits")
        assert not ref_counts(case, 3, False).any()


# ---- the kernel ----------------------------------------------------------------------------------------------------------------
@gpu
def test_variant_matrix_mixed(ctx):
    case = case_mixed()
    g = build(ctx, case)
    check_variants(g, case, "mixed")
    g.close()


@gpu
@pytest.mark.parametrize("layout", ["blocks", "interleaved"])
def test_candidate_runs_at_round_edges(ctx, layout):
    case = case_rounds(layout)
    g = build(ctx, case)
    check_variants(g, case, f"rounds {layout}")
    g.close()


@gpu
def test_nonhitting_candidates(ctx):
    case = case_nonhit()
    g = build(ctx, case)
    check_variants(g, case, "nonhit")
    g.close()


def bin_sizes(values, shift):
    return np.bincount(np.asarray(values, np.int64) >> shift)


@gpu
@pytest.mark.parametrize("regime", ["lb_cluster", "lb_shared", "lb_plateau", "lb_dense"])
def test_lower_bound_ranges(ctx, regime):
    """Databases whose LUT bins hold up to tens of thousands of records, so lb_warp's 32-probe narrowing runs for one, two and
    three steps and ends on ranges of every size; the regime is asserted through the shift the build chose."""
    case = CASES[regime]()
    g = build(ctx, case)
    shift = g.info()["lut_shift"]
    assert shift == expected_shift(case), (regime, shift)
    rc, rs, re, _ = kept_records(case)
    on0 = rc == 0
    starts = np.sort(rs[on0])
    pmax = np.maximum.accumulate(re[on0][np.argsort(rs[on0], kind="stable")])
    if regime == "lb_cluster":
        assert shift >= 15 and bin_sizes(starts, shift)[0] >= 20_000 and bin_sizes(pmax, shift)[0] >= 20_000, shift
    elif regime == "lb_shared":
        assert shift == 6
        assert set(SHARED_COUNTS) <= set(bin_sizes(starts, shift).tolist())
    elif regime == "lb_plateau":
        assert bin_sizes(pmax, shift).max() > 5000, shift
    else:
        assert shift == 0
        assert set(DENSE_COUNTS) <= set((bin_sizes(starts, 0) - 1).tolist())  # the group plus the background record
    check_variants(g, case, regime)
    g.close()


@gpu
@pytest.mark.parametrize("name", ["int32", "int32_high_shift"])
def test_int32_semantics(ctx, name):
    case = CASES[name]()
    g = build(ctx, case)
    info = g.info()
    extra = case.n_chroms - 3
    assert info["n_records"] == INT32_KEPT + extra == len(kept_records(case)[0]), info
    assert info["lut_shift"] == expected_shift(case), info
    if extra:
        assert info["lut_shift"] >= 25, info
    check_variants(g, case, name)
    g.close()


@gpu
def test_psame_across_rounds_and_m_order(ctx):
    """On one fresh database, m = 2, 5, 2, 1, 5, 3 in this order: the psame array of every new m is built inside its first
    count_region_hits call and cached; every call equals the oracle."""
    case = case_psame()
    g = build(ctx, case)
    o = make_oracle(case)
    for step, m in enumerate(case.ms):
        for binary in (True, False):
            want = oracle_counts(o, case, m, binary)
            assert_counts(ref_counts(case, m, binary), want, f"psame ref, call {step} m={m}")
            assert_counts(device_counts(g, case, m, binary), want, f"psame: call {step} (m={m}, binary={binary})")
    with knobs({"GTGPU_IGD_NO_M1": "1"}):
        assert_counts(device_counts(g, case, 1, True), oracle_counts(o, case, 1, True), "psame: general kernel at m=1")
    # every fixed query holds a 10-bp hit of each of files 1..6: whichever record is a file's first hit, it counts once
    hits = device_counts(g, case, 5, True)
    assert (hits[0, 1:7] == case.so[1]).all(), hits[0]
    g.close()


@gpu
@pytest.mark.parametrize("name", ["wide_files", "wide_chroms"])
def test_wide_build_shapes(ctx, name):
    case = CASES[name]()
    g = build(ctx, case)
    assert g.info()["n_records"] == len(kept_records(case)[0])
    check_variants(g, case, name, grids=GRIDS[:1])
    g.close()


# ---- gtgpu_igd_count_dev on device arrays ------------------------------------------------------------------------------------
def count_dev(g, set_of, qc, qs, qe, m, binary, prefill):
    """gtgpu_igd_count_dev on torch device copies of the arrays into a device matrix holding `prefill`; returns the matrix."""
    import torch
    from gtars_b200 import ffi
    dev = torch.device("cuda", 0)
    t = [torch.from_numpy(np.ascontiguousarray(a, np.uint32).view(np.int32)).to(dev) for a in (set_of, qc, qs, qe)]
    d_out = torch.from_numpy(prefill.astype(np.uint64).view(np.int64).ravel()).to(dev)
    torch.cuda.synchronize()
    ffi.check(ffi.lib().gtgpu_igd_count_dev(g._h, 1 if binary else 0, len(qc), t[0].data_ptr(), t[1].data_ptr(), t[2].data_ptr(),
                                            t[3].data_ptr(), m, d_out.data_ptr()))
    g.ctx.synchronize()
    return d_out.cpu().numpy().view(np.uint64).reshape(prefill.shape)


def sub_case(case, set_of, n_sets, idx):
    """The queries idx of case, query idx[j] in set set_of[j], grouped by set (stable) for the references."""
    order = np.argsort(set_of, kind="stable")
    sel = idx[order]
    return types.SimpleNamespace(**{**vars(case), "so": offsets(np.bincount(set_of, minlength=n_sets)),
                                    "qc": case.qc[sel], "qs": case.qs[sel], "qe": case.qe[sel]})


@gpu
def test_count_dev_accumulates_small_and_strided(ctx):
    """d_out is added to, not overwritten; n = 1..9 queries; n one more than the grid's warps at one block per SM; unsorted
    set ids; a binary call at an m no earlier call built psame for."""
    import torch
    case = case_mixed()
    g = build(ctx, case)
    o = make_oracle(case)
    rng = rng_for("count_dev")
    n_files = len(case.fo) - 1
    live = np.flatnonzero((case.qc < case.n_chroms) & (case.qs < case.qe))
    n_sets = 5
    warps = torch.cuda.get_device_properties(0).multi_processor_count * WARPS_PER_BLOCK
    sizes = list(range(1, 10)) + [warps + 1, 2000]
    for i, n in enumerate(sizes):
        idx = rng.choice(live, n, replace=n > len(live))
        set_of = rng.integers(0, n_sets, n).astype(np.uint32)
        sub = sub_case(case, set_of, n_sets, idx)
        prefill = rng.integers(0, 2**40, (n_sets, n_files)).astype(np.uint64)
        # m = 7 and m = 9 are first used here, by a binary call: psame is built inside the call
        for m, binary in ((1, False), (1, True), (2, True), (7 + (i % 2) * 2, True)):
            want = oracle_counts(o, sub, m, binary)
            assert_counts(ref_counts(sub, m, binary), want, f"count_dev ref n={n} m={m}")
            for gname, genv in GRIDS:
                with knobs(genv):
                    got = count_dev(g, set_of, case.qc[idx], case.qs[idx], case.qe[idx], m, binary, prefill)
                assert_counts(got - prefill, want, f"count_dev: n={n} m={m} binary={binary}, {gname}")
    g.close()


# ---- two devices ---------------------------------------------------------------------------------------------------------------
@gpu
def test_two_devices_match_one(ctx):
    """A database sharded by file over two devices (39 / 40 files: an unequal split) counts what one device counts."""
    from gtars_b200 import ffi
    if ffi.device_count() < 2:
        pytest.skip("needs two devices")
    multi = ffi.Context(devices=[0, 1])
    try:
        for name in ("lb_cluster", "int32"):
            case = CASES[name]()
            if (len(case.fo) - 1) % 2 == 0:  # an odd file count splits unequally
                case.fo = np.append(case.fo, case.fo[-1]).astype(np.uint64)
            one, two = build(ctx, case), build(multi, case)
            for m in case.ms:
                for binary in (False, True):
                    assert_counts(device_counts(two, case, m, binary), device_counts(one, case, m, binary),
                                  f"{name}: two devices vs one, m={m} binary={binary}")
            one.close()
            two.close()
    finally:
        multi.close()
