"""The device-resident find path called directly: gtgpu_find_dev, gtgpu_count_dev and gtgpu_unk_rule_dev on device arrays.

The fused count -> scan -> look-back -> emit kernel has template variants (Bits / AIList, min_overlap filter, per-query
offsets, lean / full kernel) and runtime paths (per-file offsets, emission cut at ids_capacity, the three warp-scan packing
regimes, file boundaries, blocks that run many tiles, the 64-bit look-back) that the host entry points only partly reach.
Every output of every call is compared with one oracle.Index.find(qc, qs, qe, m) -> (off, vals):

    ids = vals,  per-query offsets = off,  raw per-file offsets = off[file_offsets],  total = off[-1],

and the counting kernel on the same device arrays must give np.diff(off).  Output buffers start out filled with sentinels, so
a missing write shows, and the id buffer carries a guard band past its capacity, so a write past it shows too.
"""
import types
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

# Kernel geometry (kernels.cu): a tile is FUSED_BLOCK (256) threads x FUSED_ROWS (4) queries, and FUSED_SUPER tiles share
# one look-back accumulator word.  Inside a tile, warp w owns queries [128 w, 128 w + 128); query 32 row + lane of a warp
# sits in lane `lane`, row `row`.
TILE = 1024
SUPER = 64
WARP = 128
SENT32 = 0xA5A5A5A5
SENT64 = 0xA5A5A5A5A5A5A5A5
KINDS = pytest.mark.parametrize("kind", [0, 1], ids=["bits", "ailist"])
KERNELS = pytest.mark.parametrize("kernel", ["lean", "full"])

# Nested intervals on one extra chromosome that no query names: they give the index pool-list windows, so the full kernel
# serves it, with exactly the hits of the index without them.
NEST_S = np.array([1000, 2000, 2500, 10_000, 10_100], np.uint32)
NEST_E = np.array([50_000, 3000, 2600, 20_000, 10_200], np.uint32)
NEST_VAL0 = 0x40000000


# ---- harness ---------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def env():
    """One context on a torch stream: every fill, copy and library call of this module is ordered on that stream."""
    import torch
    from gtars_b200 import ffi
    stream = torch.cuda.Stream()
    ctx = ffi.Context(0, stream=stream.cuda_stream)
    yield types.SimpleNamespace(ctx=ctx, stream=stream)
    stream.synchronize()
    ctx.close()


@pytest.fixture(scope="module")
def std():
    """A clean 100 k-peak hg38-shaped universe and 300 k narrow queries sorted like one BED file."""
    from gtars_b200 import synth
    u = synth.make_universe(100_000)
    arrays = (u["chrom_offsets"].numpy().astype(np.uint64),) + tuple(u[k].numpy().view(np.uint32)
                                                                      for k in ("g_start", "g_end", "g_val"))
    q = synth.make_query_files(u, 1, 300_000)
    qc, qs, qe = (q[k].numpy().view(np.uint32).copy() for k in ("chr", "start", "end"))
    return types.SimpleNamespace(u=u, arrays=arrays, qc=qc, qs=qs, qe=qe, unk_id=int(u["unk_id"]))


def make_index(env, kind, arrays, kernel=None):
    """(device index, oracle index) over chromosome-grouped arrays.  kernel="full" appends the nested chromosome; with a
    kernel named, the index must be one that kernel serves."""
    from gtars_b200 import ffi
    from oracle import oracle as orc
    offs, s, e, v = arrays
    if kernel == "full":
        offs = np.append(offs, offs[-1] + len(NEST_S)).astype(np.uint64)
        s, e = np.concatenate([s, NEST_S]), np.concatenate([e, NEST_E])
        v = np.concatenate([v, NEST_VAL0 + np.arange(len(NEST_S), dtype=np.uint32)])
    ix = ffi.Index(env.ctx, kind, offs, s, e, v)
    ix.stream = env.stream
    if kernel is not None:
        info = ix.info()
        assert info["lean_kernel"] == (kernel == "lean") and not info["lean_fell_back"], info
    return ix, orc.Index(kind, offs, s, e, v)


def assert_ran(ix, kernel):
    """The launches so far ran `kernel` and nothing else: the lean kernel never fell back to the full one."""
    info = ix.info()
    assert info["lean_kernel"] == (kernel == "lean") and not info["lean_fell_back"], info


def oracle_find(o, qc, qs, qe, m=0):
    """oracle.Index.find, split over threads for large batches (ctypes releases the GIL; the oracle index is read-only)."""
    n = len(qc)
    if n <= 1 << 20:
        return o.find(qc, qs, qe, m)
    cuts = np.linspace(0, n, 17).astype(np.int64)
    spans = list(zip(cuts[:-1], cuts[1:]))
    with ThreadPoolExecutor(len(spans)) as ex:
        parts = list(ex.map(lambda ab: o.find(qc[ab[0]:ab[1]], qs[ab[0]:ab[1]], qe[ab[0]:ab[1]], m), spans))
    off = np.empty(n + 1, np.uint64)
    base = 0
    for (a, b), (po, _) in zip(spans, parts):
        off[a:b] = po[:-1] + np.uint64(base)
        base += int(po[-1])
    off[n] = base
    return off, np.concatenate([pv for _, pv in parts])


def _dev(a, dtype):
    import torch
    a = np.ascontiguousarray(a, dtype=dtype)
    return torch.from_numpy(a.view(np.int32 if a.itemsize == 4 else np.int64)).to("cuda")


def _filled(n, wide=False):
    import torch
    if wide:
        return torch.full((n,), SENT64 - (1 << 64), dtype=torch.int64, device="cuda")
    return torch.full((n,), SENT32 - (1 << 32), dtype=torch.int32, device="cuda")


def _host(t, dtype):
    return t.cpu().numpy().view(dtype)


def _ptr(t):
    return t.data_ptr() if t is not None else None


def run_find_dev(ix, qc, qs, qe, min_overlap, file_offsets=None, per_query=True, capacity=None, guard=4096, ids=True,
                 id_shift=0, fetch_ids=True):
    """Uploads the queries, runs gtgpu_count_dev and then gtgpu_find_dev on them, and returns every output.

    The id buffer holds id_shift + capacity + guard sentinel words and find_dev writes from word id_shift on (capacity None:
    the sum of count_dev's counts); offsets start as sentinels too.  ids=False is the ABI's no-output form: d_out_ids NULL,
    ids_capacity 0.  Returns ids (the whole buffer, head and guard included, unless fetch_ids is False), offsets, raw per-file
    offsets, total and the per-query counts of count_dev; d_ids / d_file_tok stay on the device for chained calls."""
    import torch
    n = len(qc)
    with torch.cuda.stream(ix.stream):
        d_c, d_s, d_e = (_dev(a, np.uint32) for a in (qc, qs, qe))
        d_counts = _filled(max(n, 1))
        ix.count_dev(n, d_c.data_ptr(), d_s.data_ptr(), d_e.data_ptr(), min_overlap, d_counts.data_ptr())
        counts = _host(d_counts[:n], np.uint32)  # a synchronous copy on the stream
        if capacity is None:
            capacity = int(counts.sum(dtype=np.uint64)) if ids else 0
        d_ids = _filled(id_shift + capacity + guard) if ids else None
        d_off = _filled(n + 1, True) if per_query else None
        d_fo = d_ftok = None
        n_files = 0
        if file_offsets is not None:
            n_files = len(file_offsets) - 1
            d_fo = _dev(file_offsets, np.uint64)
            d_ftok = _filled(n_files + 1, True)
        d_total = _filled(1, True)
        ix.find_dev(n, d_c.data_ptr(), d_s.data_ptr(), d_e.data_ptr(), min_overlap, n_files, _ptr(d_fo),
                    d_ids.data_ptr() + 4 * id_shift if ids else None, capacity if ids else 0, _ptr(d_off), _ptr(d_ftok),
                    d_total.data_ptr())
        ix.stream.synchronize()
        return types.SimpleNamespace(
            cap=capacity if ids else 0, shift=id_shift, d_ids=d_ids, d_file_tok=d_ftok, counts=counts,
            total=int(_host(d_total, np.uint64)[0]),
            offsets=_host(d_off, np.uint64) if per_query else None,
            file_tok=_host(d_ftok, np.uint64) if d_ftok is not None else None,
            ids=_host(d_ids, np.uint32) if ids and fetch_ids else None)


def assert_same(got, want, what):
    got, want = np.asarray(got), np.asarray(want)
    assert got.shape == want.shape, f"{what}: {got.shape} != {want.shape}"
    bad = np.flatnonzero(got != want)
    assert len(bad) == 0, (f"{what}: {len(bad)} of {len(want)} differ, first at {bad[0]}: "
                           f"got {got[bad[0]]:#x}, want {want[bad[0]]:#x}")


def check(r, exp, file_offsets=None):
    """Every output of run_find_dev against the oracle's (off, vals); vals may stop after min(capacity, total)."""
    off, vals = exp
    total = int(off[-1])
    assert r.total == total
    assert_same(r.counts, np.diff(off).astype(np.uint32), "count_dev")
    if r.offsets is not None:
        assert_same(r.offsets, off, "per-query offsets")
    if r.file_tok is not None:
        assert_same(r.file_tok, off[np.asarray(file_offsets, np.int64)], "per-file offsets")
    if r.ids is not None:
        k = min(r.cap, total)
        body = r.ids[r.shift:]
        assert_same(body[:k], vals[:k], "ids")
        assert (r.ids[:r.shift] == SENT32).all(), "written before the id buffer"
        assert_same(body[k:], np.full(len(body) - k, SENT32, np.uint32), "past min(total, capacity)")


def ragged_files(n, n_files, seed):
    """File offsets over n queries: random sizes, some empty files, an empty first and last file."""
    rng = np.random.default_rng(seed)
    cuts = np.sort(rng.integers(0, n + 1, n_files - 3))
    cuts[1::13] = cuts[0::13][:len(cuts[1::13])]  # some empty files
    return np.concatenate([[0, 0], cuts, [n, n]]).astype(np.uint64)


def run_unk_rule(env, n_files, d_raw_tok, d_raw_ids, raw_total, unk_id, guard=1024):
    """gtgpu_unk_rule_dev into sentinel-filled outputs: (token offsets, id buffer with guard, n_empty)."""
    import torch
    with torch.cuda.stream(env.stream):
        d_tok = _filled(n_files + 1, True)
        d_ids = _filled(raw_total + n_files + guard)
        d_n = _filled(1, True)
        env.ctx.unk_rule_dev(n_files, d_raw_tok.data_ptr(), d_raw_ids.data_ptr(), unk_id, d_tok.data_ptr(), d_ids.data_ptr(),
                             d_n.data_ptr())
        env.stream.synchronize()
        return _host(d_tok, np.uint64), _host(d_ids, np.uint32), int(_host(d_n, np.uint64)[0])


def check_unk(got, want_tok, want_ids, want_empty):
    tok, ids, n_empty = got
    assert_same(tok, want_tok, "token offsets")
    assert_same(ids[:len(want_ids)], want_ids, "token ids")
    assert (ids[len(want_ids):] == SENT32).all(), "written past the token ids"
    assert n_empty == want_empty


# ---- 1. every variant ------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("m", [0, 1, 2, 37])
@KERNELS
@KINDS
def test_variant_matrix(env, std, kind, kernel, m):
    """Bits / AIList x lean / full x min_overlap x per-query offsets on / off x per-file offsets on / off, and the form without
    any output but the total."""
    ix, o = make_index(env, kind, std.arrays, kernel)
    n = 200_000
    qc, qs, qe = std.qc[:n], std.qs[:n], std.qe[:n]
    fo = ragged_files(n, 300, seed=m)
    exp = o.find(qc, qs, qe, m)
    for per_query in (False, True):
        for files in (None, fo):
            check(run_find_dev(ix, qc, qs, qe, m, files, per_query), exp, files)
            assert_ran(ix, kernel)
    check(run_find_dev(ix, qc, qs, qe, m, per_query=False, ids=False), exp)
    assert_ran(ix, kernel)
    if m == 37:
        assert int(exp[0][-1]) < int(o.find(qc, qs, qe, 0)[0][-1])  # the filter removed hits


# ---- 2. query counts around warp, tile and supertile sizes -----------------------------------------------------------------
@KERNELS
@KINDS
def test_query_count_shapes(env, std, kind, kernel):
    ix, o = make_index(env, kind, std.arrays, kernel)
    for n in (0, 1, 31, 32, 127, 128, 1023, 1024, 1025, 2048, 65535, 65536, 65537, 3 * 65536 + 1):
        qc, qs, qe = std.qc[:n], std.qs[:n], std.qe[:n]
        fo = np.array([0, n // 3, n // 3, n // 2, n], np.uint64)
        r = run_find_dev(ix, qc, qs, qe, 0, fo)
        if n == 0:
            assert r.offsets[0] == 0 and (r.file_tok == 0).all() and r.total == 0
        check(r, o.find(qc, qs, qe), fo)
    assert_ran(ix, kernel)


# ---- 3. exact hit multiplicities per warp ----------------------------------------------------------------------------------
STACKS = (1, 2, 3, 4, 5, 6, 7, 8, 15, 16, 20, 300, 1500)


def stack_universe():
    """Chromosome 0 holds, for each c in STACKS, a stack of c intervals at P = 10^6 (j + 1):
    interval i = [P + i % 100, P + 101 + 37 i % 100).  The query [P + 100, P + 200) hits all c of them, with 1 + 37 i % 100 bp
    of overlap, so a min_overlap removes a known part.  Stacks of 3-15 give pool-list windows, larger ones overflow windows."""
    s, e, pos = [], [], {}
    for j, c in enumerate(STACKS):
        p = 1_000_000 * (j + 1)
        pos[c] = p
        i = np.arange(c)
        s.append(p + i % 100)
        e.append(p + 101 + (37 * i) % 100)
    s, e = np.concatenate(s).astype(np.uint32), np.concatenate(e).astype(np.uint32)
    return (np.array([0, len(s)], np.uint64), s, e, np.arange(len(s), dtype=np.uint32)), pos


def pair_universe():
    """A clean universe (the lean kernel serves it): pairs [P, P + 150), [P + 140, P + 300) that overlap without nesting,
    and single intervals; the query [P + 100, P + 200) hits 2 (overlaps 50 and 60 bp) or 1."""
    s = np.array([100_000, 100_140, 300_000], np.uint32)
    e = np.array([100_150, 100_300, 300_150], np.uint32)
    return (np.array([0, 3], np.uint64), s, e, np.array([7, 11, 13], np.uint32)), {2: 100_000, 1: 300_000}


def layout_queries(counts, pos):
    """One query per entry of `counts` (query order), each with exactly that many hits at min_overlap 0."""
    counts = np.asarray(counts)
    p = np.array([pos.get(int(c), 0) for c in counts], np.int64)
    qs = np.where(counts == 0, 500 + np.arange(len(counts)) % 1000, p + 100).astype(np.uint32)
    return np.zeros(len(counts), np.uint32), qs, qs + 100


def warps(*ws):
    """Concatenates warp layouts: each a scalar count for all 128 queries or a 128-entry array (index = 32 row + lane)."""
    return np.concatenate([np.full(WARP, w) if np.isscalar(w) else np.asarray(w) for w in ws])


def regime_layout(seed):
    rng = np.random.default_rng(seed)
    small = [0, 1, 2, 3, 4, 5, 6, 7]
    seven_eight = np.full(WARP, 7)
    seven_eight[127] = 8  # lane 31 of row 3: one hit past WARP_SEMI
    w300 = rng.choice([0, 1, 2], WARP)
    w300[5] = 300  # past 8-bit offsets
    w1500 = rng.choice([0, 1, 2], WARP)
    w1500[64] = 1500  # past 10-bit row bases
    tiles = [
        warps(*[2] * 8),                # bytewise scan at its maximum: row sums 64, packed offsets up to 254
        warps(*[7] * 8),                # WARP_SEMI at its maximum: row sums 224, row bases 224 / 448 / 672
        warps(*[seven_eight] * 8),      # one query past it: WARP_SLOW
        warps(2, 7, seven_eight, 0, 1, rng.choice(small, WARP), rng.choice([0, 1, 2, 7, 8, 15, 16, 20], WARP), 2),
        warps(w300, w1500, 7, rng.choice(small, WARP), 2, 0, rng.choice(small + [16], WARP), 7),
        rng.choice(small + [16], 300),  # a partial last tile
    ]
    return np.concatenate(tiles)


@KINDS
def test_warp_regimes_exact_multiplicities(env, kind):
    """Whole warps with every count 2, every count 7, 127 x 7 + one 8, single queries with 300 and 1 500 hits, and warps of
    one tile in different regimes (full kernel: the universe has pool and overflow windows)."""
    arrays, pos = stack_universe()
    ix, o = make_index(env, kind, arrays)
    assert not ix.info()["lean_kernel"]
    counts = regime_layout(seed=kind)
    qc, qs, qe = layout_queries(counts, pos)
    n = len(qc)
    fo = np.array([0, TILE, 1500, 3 * TILE, 3 * TILE, n], np.uint64)
    for m in (0, 50):
        exp = o.find(qc, qs, qe, m)
        if m == 0:
            assert_same(np.diff(exp[0]), counts.astype(np.uint64), "hits by construction")
        else:
            assert int(exp[0][-1]) < int(counts.sum())
        check(run_find_dev(ix, qc, qs, qe, m, fo), exp, fo)


@KINDS
def test_lean_two_hit_warps(env, kind):
    """The lean kernel's bytewise scan at its maximum (every count 2) and the AIList two-hit order, whole tiles of it."""
    arrays, pos = pair_universe()
    ix, o = make_index(env, kind, arrays, "lean")
    counts = np.concatenate([warps(*[2] * 8), warps(*[1] * 8), warps(2, 1, 0, 2, 2, 1, 2, 2), np.full(77, 2)])
    qc, qs, qe = layout_queries(counts, pos)
    fo = np.array([0, 1000, 2 * TILE, len(qc)], np.uint64)
    for m in (0, 55):
        exp = o.find(qc, qs, qe, m)
        if m == 0:
            assert_same(np.diff(exp[0]), counts.astype(np.uint64), "hits by construction")
        check(run_find_dev(ix, qc, qs, qe, m, fo), exp, fo)
    assert_ran(ix, "lean")


# ---- 4. ids_capacity -------------------------------------------------------------------------------------------------------
def capacity_cases(off, extra=()):
    total = int(off[-1])
    n = len(off) - 1
    t = (n // TILE) // 2
    caps = {total, total - 1, int(off[min(n, TILE) // 2]) + 1, int(off[t * TILE + 517]) + 1, int(off[t * TILE]), 0}
    return sorted(c for c in caps.union(extra) if 0 <= c <= total)


def _check_capacities(ix, o, qc, qs, qe, fo, extra=()):
    exp = o.find(qc, qs, qe)
    for cap in capacity_cases(exp[0], extra):
        # totals and offsets do not depend on the capacity; ids below it are exact, nothing lands past it
        check(run_find_dev(ix, qc, qs, qe, 0, fo, capacity=cap), exp, fo)


@KERNELS
@KINDS
def test_capacity_cuts(env, std, kind, kernel):
    ix, o = make_index(env, kind, std.arrays, kernel)
    n = 50 * TILE + 300
    qc, qs, qe = std.qc[:n], std.qs[:n], std.qe[:n]
    _check_capacities(ix, o, qc, qs, qe, ragged_files(n, 40, seed=4))
    assert_ran(ix, kernel)


@KINDS
def test_capacity_cuts_warp_regimes(env, kind):
    """Capacity cuts on the full kernel with WARP_SEMI / WARP_SLOW warps, one inside the 1 500-hit query's run."""
    arrays, pos = stack_universe()
    ix, o = make_index(env, kind, arrays)
    counts = regime_layout(seed=kind)
    qc, qs, qe = layout_queries(counts, pos)
    q1500 = int(np.flatnonzero(counts == 1500)[0])
    off = np.concatenate([[0], np.cumsum(counts)])
    _check_capacities(ix, o, qc, qs, qe, np.array([0, 2000, len(qc)], np.uint64), extra=(int(off[q1500]) + 700,))


# ---- 5. file boundaries ----------------------------------------------------------------------------------------------------
def file_layouts():
    n1 = 10 * TILE + 300
    n3 = 8 * TILE + 5
    q0 = 3 * TILE + 10
    n5 = 4 * SUPER * TILE
    return {
        "tile_starts": (n1, np.arange(0, n1, TILE).tolist() + [n1]),
        "n_multiple_of_tile": (8 * TILE, [0, 100, 5000, 8 * TILE]),
        "crowded_tile": (n3, [0] + [q0 + i for i in range(300)] + [q0 + 300] * 5000 + [n3]),
        "empty_at_0_and_n": (n1, [0] * 50 + [500, 7000] + [n1] * 50),
        "three_supertiles": (n5, [0, 1000, 1000 + 3 * SUPER * TILE + 5, n5]),
        "no_files": (5000, [0]),
    }


@KERNELS
@KINDS
def test_file_boundaries_and_unk_rule(env, std, kind, kernel):
    """Raw per-file offsets at tile starts, at n = 8 x 1 024, 300 + 5 000 boundaries in one tile, empty files at 0 and n, one
    file over three supertiles and no file at all; then gtgpu_unk_rule_dev on those raw outputs against tokenize_files."""
    ix, o = make_index(env, kind, std.arrays, kernel)
    for name, (n, fo) in file_layouts().items():
        fo = np.array(fo, np.uint64)
        qc, qs, qe = std.qc[:n], std.qs[:n], std.qe[:n]
        r = run_find_dev(ix, qc, qs, qe, 0, fo)
        check(r, o.find(qc, qs, qe), fo)
        want_tok, want_ids = o.tokenize_files(fo, qc, qs, qe, std.unk_id)
        got = run_unk_rule(env, len(fo) - 1, r.d_file_tok, r.d_ids, r.total, std.unk_id)
        check_unk(got, want_tok, want_ids, int((np.diff(r.file_tok) == 0).sum()))
    assert_ran(ix, kernel)


# ---- 6. gtgpu_unk_rule_dev alone -------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n_files", [0, 1, 1023, 1024, 1025, 5000])
def test_unk_rule_dev(env, n_files):
    """One block of 1 024 threads loops over the files: empty-file counts must carry from one pass to the next."""
    rng = np.random.default_rng(n_files)
    unk = 0x7FFF0001
    f = np.arange(n_files)
    for pattern in ("none", "all", "alternating", "runs"):
        cnt = rng.integers(1, 4, n_files)
        if pattern == "all":
            cnt[:] = 0
        elif pattern == "alternating":
            cnt[f % 2 == 1] = 0
        elif pattern == "runs":  # runs of empty files across the 1 024 and 2 048 boundaries, at the start and the end
            cnt[(f < 5) | ((f >= 1000) & (f < 1100)) | ((f >= 2040) & (f < 2060)) | (f >= n_files - 30)] = 0
        raw = np.concatenate([[0], np.cumsum(cnt)]).astype(np.uint64)
        raw_ids = rng.integers(0, 1 << 31, int(raw[-1])).astype(np.uint32)
        empty = cnt == 0
        want_tok = raw + np.concatenate([[0], np.cumsum(empty)]).astype(np.uint64)
        want_ids = np.concatenate([[np.uint32(unk)] if empty[i] else raw_ids[raw[i]:raw[i + 1]] for i in range(n_files)]
                                  + [np.zeros(0, np.uint32)]).astype(np.uint32)
        got = run_unk_rule(env, n_files, _dev(raw, np.uint64), _dev(np.append(raw_ids, np.uint32(0)), np.uint32), int(raw[-1]),
                           unk)
        check_unk(got, want_tok, want_ids, int(empty.sum()))


# ---- 7. blocks that run many tiles -----------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def big(std):
    """64 tiles per SM and a partial last tile (~10 M queries on 148 SMs), ragged files, 1 % unknown chromosomes and 1 %
    empty queries (placed where the lean kernel's window test still holds)."""
    import torch
    from gtars_b200 import synth
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    n = 64 * sms * TILE + 517
    q = synth.make_query_files(std.u, 1, n, device="cuda", unknown_frac_ppm=10_000)
    qc, qs, qe = (q[k].cpu().numpy().view(np.uint32).copy() for k in ("chr", "start", "end"))
    rng = np.random.default_rng(7)
    deg = rng.choice(n, n // 100, replace=False)
    qs[deg] |= 1
    qe[deg] = qs[deg]
    return types.SimpleNamespace(n=n, qc=qc, qs=qs, qe=qe, fo=ragged_files(n, 2000, seed=7), exp={})


@KERNELS
@KINDS
def test_many_tiles_per_block(env, std, big, kind, kernel):
    """Persistent blocks run many tiles (lag-1 pipeline, parity double buffers): full oracle comparison, and a second run
    hands the tiles out in another order but must give identical bytes."""
    ix, o = make_index(env, kind, std.arrays, kernel)
    if kind not in big.exp:
        big.exp[kind] = oracle_find(o, big.qc, big.qs, big.qe)
    r1 = run_find_dev(ix, big.qc, big.qs, big.qe, 0, big.fo)
    check(r1, big.exp[kind], big.fo)
    r2 = run_find_dev(ix, big.qc, big.qs, big.qe, 0, big.fo)
    assert_same(r2.ids, r1.ids, "ids, second run")
    assert_same(r2.offsets, r1.offsets, "per-query offsets, second run")
    assert_same(r2.file_tok, r1.file_tok, "per-file offsets, second run")
    assert_ran(ix, kernel)


# ---- 8. one query sends the lean kernel to its fallback --------------------------------------------------------------------
@pytest.mark.parametrize("where", ["query_0", "lane31_row3_mid_tile", "last_of_partial_tile"])
@KINDS
def test_lean_fallback_from_one_query(env, std, kind, where):
    n = 300_000  # 292 full tiles and a partial one
    qc, qs, qe = std.qc[:n].copy(), std.qs[:n].copy(), std.qe[:n].copy()
    i = {"query_0": 0, "lane31_row3_mid_tile": 150 * TILE + 5 * WARP + 3 * 32 + 31, "last_of_partial_tile": n - 1}[where]
    if where == "lane31_row3_mid_tile":
        qc[i], qs[i], qe[i] = 0, 5_000_123, 5_000_123 - 50_000  # reversed
    else:
        qc[i], qs[i], qe[i] = 0, 5_000_000, 5_300_000  # wide
    ix, o = make_index(env, kind, std.arrays, "lean")  # fresh: the fallback is remembered per index
    fo = ragged_files(n, 100, seed=8)
    check(run_find_dev(ix, qc, qs, qe, 0, fo), o.find(qc, qs, qe), fo)
    info = ix.info()
    assert info["lean_kernel"] and info["lean_fell_back"], info


# ---- 9. totals and id positions past 2^32 ----------------------------------------------------------------------------------
K_STACK = 5000
N_STACK = 1_000_000


def huge_case(env, kind):
    """K identical intervals on chromosome 0 and N queries inside them: query i owns ids [i K, i K + K), K N ~ 5e9."""
    s = np.full(K_STACK, 1000, np.uint32)
    e = np.full(K_STACK, 3_000_000, np.uint32)
    ix, o = make_index(env, kind, (np.array([0, K_STACK], np.uint64), s, e, np.arange(K_STACK, dtype=np.uint32)))
    i = np.arange(N_STACK, dtype=np.uint64)
    qc = np.zeros(N_STACK, np.uint32)
    qs = (2000 + (i * 7919) % 2_000_000).astype(np.uint32)
    qe = qs + 50
    ref = o.find(qc[:1], qs[:1], qe[:1])[1]
    assert len(ref) == K_STACK
    return ix, (qc, qs, qe), ref, i


@KINDS
def test_total_past_2_32(env, kind):
    ix, (qc, qs, qe), ref, i = huge_case(env, kind)
    off = np.append(i, np.uint64(N_STACK)) * np.uint64(K_STACK)
    assert int(off[-1]) > 1 << 32
    fo = np.array([0, 1, 2, 1000, 500_000, N_STACK], np.uint64)
    cap = 3 * K_STACK + 123
    r = run_find_dev(ix, qc, qs, qe, 0, fo, capacity=cap)
    check(r, (off, np.tile(ref, 4)), fo)


def test_id_positions_past_2_32(env):
    """Capacity just above 2^32 ids (17 GB), the id buffer starting at an odd word: ids around position 2^32 are exact."""
    import torch
    free, _ = torch.cuda.mem_get_info()
    if free < 24 << 30:
        pytest.skip(f"needs about 24 GB of free device memory, {free >> 30} GB free")
    ix, (qc, qs, qe), ref, i = huge_case(env, 0)
    cap, shift = (1 << 32) + (1 << 20), 3
    r = run_find_dev(ix, qc, qs, qe, 0, capacity=cap, id_shift=shift, guard=1 << 16, fetch_ids=False)
    off = np.append(i, np.uint64(N_STACK)) * np.uint64(K_STACK)
    check(r, (off, None))
    w = 1 << 16
    for lo in ((1 << 32) - w, cap - w):
        got = _host(r.d_ids[shift + lo:shift + lo + w], np.uint32)
        assert_same(got, ref[np.arange(lo, lo + w, dtype=np.uint64) % np.uint64(K_STACK)], f"ids from position {lo}")
    assert (_host(r.d_ids[:shift], np.uint32) == SENT32).all()
    assert (_host(r.d_ids[shift + cap:], np.uint32) == SENT32).all(), "written past the capacity"
    del r
    torch.cuda.empty_cache()
