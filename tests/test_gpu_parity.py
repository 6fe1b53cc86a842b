"""GPU parity: the CUDA path (through the C ABI of include/gtars_gpu.h) against the CPU oracle, bit-exact.

Run on a B200 with `pytest -m gpu`.  Inputs are seeded; sizes are chosen so the oracle finishes in seconds;
full-size properties live in test_gpu_scale.py.
"""
import zlib

import numpy as np
import pytest

from tests import helpers
from tests.helpers import KINDS

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    from gtars_b200 import ffi
    c = ffi.Context(0)
    yield c
    c.close()


def _both(ctx, kind, offs, s, e, v=None):
    from gtars_b200 import ffi
    from oracle import oracle as orc
    return ffi.Index(ctx, KINDS[kind], offs, s, e, v), orc.Index(KINDS[kind], offs, s, e, v)


def _assert_same_find(g, o, qc, qs, qe, m=0):
    go, gv = g.find(qc, qs, qe, m)
    oo, ov = o.find(qc, qs, qe, m)
    assert np.array_equal(go, oo)
    assert np.array_equal(gv, ov)
    assert np.array_equal(g.count(qc, qs, qe, m), o.count(qc, qs, qe, m))
    assert np.array_equal(g.any(qc, qs, qe, m), o.any(qc, qs, qe, m))


# ---- the reference's own KATs, replayed through the C ABI --------------------------------------------------------
@pytest.mark.parametrize("name", ["K1_abcd", "K1_empty", "K1_single", "K2_nested26"])
def test_overlapper_kats_gpu(ctx, golden, name):
    case = golden[1][name]
    ivs = case["intervals"]
    offs = np.array([0, len(ivs)], dtype=np.uint64)
    s = np.array([iv[0] for iv in ivs], dtype=np.uint32)
    e = np.array([iv[1] for iv in ivs], dtype=np.uint32)
    for kind in case["kinds"]:
        g, o = _both(ctx, kind, offs, s, e)
        if kind == "ailist" and "ailist_components" in case:
            assert g.info()["max_components"] == case["ailist_components"]
        for q in case["queries"]:
            qc = np.zeros(1, dtype=np.uint32)
            qs = np.array([q["q"][0]], dtype=np.uint32)
            qe = np.array([q["q"][1]], dtype=np.uint32)
            off, vals = g.find(qc, qs, qe)
            got = sorted((int(s[v]), int(e[v])) for v in vals)
            if "set" in q:
                assert got == sorted(tuple(x) for x in q["set"]), (name, kind, q)
            if "n" in q:
                assert len(vals) == q["n"] and g.count(qc, qs, qe)[0] == q["n"], (name, kind, q)
            _assert_same_find(g, o, qc, qs, qe)


def test_bits_count_and_order_gpu(ctx, golden):
    case = golden[1]["K3_bits_count"]
    ivs = case["intervals"]
    offs = np.array([0, len(ivs)], dtype=np.uint64)
    s = np.array([iv[0] for iv in ivs], dtype=np.uint32)
    e = np.array([iv[1] for iv in ivs], dtype=np.uint32)
    g, o = _both(ctx, "bits", offs, s, e)
    for q in case["queries"]:
        qc, qs, qe = np.zeros(1, np.uint32), np.array([q["q"][0]], np.uint32), np.array([q["q"][1]], np.uint32)
        assert g.bits_count(qc, qs, qe)[0] == q["count"]
        assert g.count(qc, qs, qe)[0] == q["find_n"]
    case = golden[1]["K3_bits_order"]
    ivs = case["intervals_val"]
    offs = np.array([0, len(ivs)], dtype=np.uint64)
    s = np.array([iv[0] for iv in ivs], dtype=np.uint32)
    e = np.array([iv[1] for iv in ivs], dtype=np.uint32)
    v = np.array([iv[2] for iv in ivs], dtype=np.uint32)
    g, o = _both(ctx, "bits", offs, s, e, v)
    for q in case["queries"]:
        qc, qs, qe = np.zeros(1, np.uint32), np.array([q["q"][0]], np.uint32), np.array([q["q"][1]], np.uint32)
        _, vals = g.find(qc, qs, qe)
        assert [int(x) for x in vals] == [t[2] for t in q["ordered"]]


@pytest.mark.parametrize("kind", ["bits", "ailist"])
def test_mco_kats_gpu(ctx, golden, kind):
    for case in golden[1]["K4_mco"]:
        cmap, offs, s, e, v = helpers.flatten_source(case["source"])
        g, o = _both(ctx, kind, offs, s, e, v)
        qc, qs, qe = helpers.flatten_queries(case["query"], cmap)
        m = case["min_overlap"] if case["min_overlap"] is not None else 0
        if "count" in case:
            assert list(g.count(qc, qs, qe, m)) == case["count"], case["cite"]
        if "any" in case:
            assert list(g.any(qc, qs, qe, m)) == case["any"], case["cite"]
        off, vals = g.find(qc, qs, qe, m)
        if "find" in case:
            src = case["source"]
            got = [sorted([src[int(x)][1], src[int(x)][2]] for x in vals[int(off[i]):int(off[i + 1])])
                   for i in range(len(qc))]
            assert got == [sorted(x) for x in case["find"]], case["cite"]
        if "find_idx" in case:
            got = [sorted(int(x) for x in vals[int(off[i]):int(off[i + 1])]) for i in range(len(qc))]
            assert got == case["find_idx"], case["cite"]
        _assert_same_find(g, o, qc, qs, qe, m)


# ---- randomized differential tests ------------------------------------------------------------------------------------
def _random_index(rng, n_chroms, n, style):
    chr_ = np.sort(rng.integers(0, n_chroms, n))
    span = 200_000
    if style == "peaks":  # non-overlapping
        s = np.empty(n, dtype=np.int64)
        e = np.empty(n, dtype=np.int64)
        for c in range(n_chroms):
            idx = np.where(chr_ == c)[0]
            k = len(idx)
            if k == 0:
                continue
            slot = max(span // k, 4)
            base = np.arange(k) * slot
            w = rng.integers(1, max(slot - 1, 2), k)
            perm = rng.permutation(k)
            s[idx] = base[perm]
            e[idx] = (base + w)[perm]
    elif style == "overlap":
        s = rng.integers(0, span, n)
        e = s + rng.integers(1, 3000, n)
    elif style == "nested":
        s = rng.integers(0, span, n)
        w = np.where(rng.random(n) < 0.08, rng.integers(5000, 60000, n), rng.integers(1, 400, n))
        e = s + w
    elif style == "dups":
        s = rng.integers(0, 500, n) * 100
        e = s + rng.integers(0, 3, n) * 150  # zero-length and duplicates
    elif style == "degenerate":
        s = rng.integers(0, span, n)
        e = s + rng.integers(-500, 2000, n)  # some start > end
        e = np.maximum(e, 0)
    else:
        raise ValueError(style)
    counts = np.bincount(chr_, minlength=n_chroms)
    offs = np.concatenate([[0], np.cumsum(counts)]).astype(np.uint64)
    return offs, s.astype(np.uint32), e.astype(np.uint32), rng.permutation(n).astype(np.uint32)


def _random_queries(rng, n_chroms, nq, degenerate=False):
    qc = rng.integers(0, n_chroms + 2, nq).astype(np.uint32)  # ids >= n_chroms are unknown
    qc[rng.random(nq) < 0.02] = 0xFFFFFFFF
    qs = rng.integers(0, 210_000, nq)
    qe = qs + rng.integers(1, 2500, nq)
    if degenerate:
        k = rng.random(nq)
        qe = np.where(k < 0.1, qs, qe)          # empty
        qe = np.where((k >= 0.1) & (k < 0.2), np.maximum(qs - rng.integers(1, 900, nq), 0), qe)  # reversed
        qs = np.where(k > 0.97, 0xFFFFFFFF, qs)
        qe = np.where(k > 0.985, 0xFFFFFFFF, qe)
    return qc, qs.astype(np.uint32), qe.astype(np.uint32)


@pytest.mark.parametrize("kind", ["bits", "ailist"])
@pytest.mark.parametrize("style", ["peaks", "overlap", "nested", "dups", "degenerate"])
def test_random_differential(ctx, kind, style):
    import zlib
    rng = np.random.default_rng(zlib.crc32(f"{kind}/{style}".encode()))
    n_chroms = 5
    offs, s, e, v = _random_index(rng, n_chroms, 6000, style)
    g, o = _both(ctx, kind, offs, s, e, v)
    if kind == "ailist" and style == "nested":
        assert g.info()["max_components"] >= 2
    for degenerate in (False, True):
        qc, qs, qe = _random_queries(rng, n_chroms, 5000, degenerate)
        for m in (0, 1, 2, 50):
            _assert_same_find(g, o, qc, qs, qe, m)
        if kind == "bits":
            assert np.array_equal(g.bits_count(qc, qs, qe), o.bits_count(qc, qs, qe))


@pytest.mark.parametrize("kind", ["bits", "ailist"])
@pytest.mark.parametrize("style", ["overlap", "nested", "dups", "degenerate"])
def test_device_sorted_build_matches_host_sorted_build(ctx, kind, style, monkeypatch):
    """gtgpu_index_build orders large inputs with stable radix passes on the device (build.cu) and small ones with the
    host's stable sort: both must give the reference's order — ties on (start, end) / start keep insertion order, which
    the duplicate-heavy styles exercise through the hits' vals — and the same search tables."""
    rng = np.random.default_rng(zlib.crc32(f"devbuild/{kind}/{style}".encode()))
    n_chroms = 7
    offs, s, e, v = _random_index(rng, n_chroms, 9000, style)
    from gtars_b200 import ffi
    monkeypatch.setenv("GTGPU_BUILD_SORT", "device")
    g_dev, o = _both(ctx, kind, offs, s, e, v)
    monkeypatch.setenv("GTGPU_BUILD_SORT", "host")
    g_host = ffi.Index(ctx, KINDS[kind], offs, s, e, v)
    i_dev, i_host = g_dev.info(), g_host.info()
    assert i_dev == i_host
    qc, qs, qe = _random_queries(rng, n_chroms, 6000, style == "degenerate")
    for m in (0, 2):
        _assert_same_find(g_dev, o, qc, qs, qe, m)
        a, b = g_dev.find(qc, qs, qe, m), g_host.find(qc, qs, qe, m)
        assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])
    if kind == "bits":
        assert np.array_equal(g_dev.bits_count(qc, qs, qe), o.bits_count(qc, qs, qe))
    # chromosomes without intervals and an empty index go through the device path too
    offs2 = np.array([0, 0, 3, 3], dtype=np.uint64)
    s2, e2 = np.array([50, 10, 10], np.uint32), np.array([60, 30, 20], np.uint32)
    monkeypatch.setenv("GTGPU_BUILD_SORT", "device")
    g2, o2 = _both(ctx, kind, offs2, s2, e2)
    q = (np.array([0, 1, 2, 1], np.uint32), np.array([0, 0, 0, 15], np.uint32), np.array([100, 100, 100, 55], np.uint32))
    _assert_same_find(g2, o2, *q)


@pytest.mark.parametrize("kind", ["bits", "ailist"])
@pytest.mark.parametrize("style", ["peaks", "overlap", "nested", "dups"])
def test_partitioned_count_matches_direct_and_oracle(ctx, kind, style, monkeypatch):
    """The bucketed counting pass (queries grouped by rank-LUT slice, used for databases beyond the L2) returns what the
    direct pass and the oracle return, for every output type, tile remainders and unknown / degenerate queries."""
    rng = np.random.default_rng(zlib.crc32(f"part/{kind}/{style}".encode()))
    n_chroms = 5
    offs, s, e, v = _random_index(rng, n_chroms, 6000, style)
    g, o = _both(ctx, kind, offs, s, e, v)
    for nq, degenerate in ((1, False), (15, True), (4095, False), (4096, True), (4097, False), (70_001, True)):
        qc, qs, qe = _random_queries(rng, n_chroms, nq, degenerate)
        monkeypatch.setenv("GTGPU_COUNT_PARTITION", "0")
        direct = g.count(qc, qs, qe), g.any(qc, qs, qe), (g.bits_count(qc, qs, qe) if kind == "bits" else None)
        monkeypatch.setenv("GTGPU_COUNT_PARTITION", "1")
        n0 = ctx.launch_count()
        part = g.count(qc, qs, qe), g.any(qc, qs, qe), (g.bits_count(qc, qs, qe) if kind == "bits" else None)
        per_call = 3 if g.info()["proper"] else 1                        # stage, count the runs, unstage
        assert ctx.launch_count() - n0 == per_call * (3 if kind == "bits" else 2)
        assert np.array_equal(part[0], o.count(qc, qs, qe))
        assert np.array_equal(part[0], direct[0]) and np.array_equal(part[1], direct[1])
        if kind == "bits":
            assert np.array_equal(part[2], o.bits_count(qc, qs, qe)) and np.array_equal(part[2], direct[2])
        assert np.array_equal(g.count(qc, qs, qe, 2), o.count(qc, qs, qe, 2))  # min_overlap > 1 never partitions


def test_bucketed_count_wide_coordinates(ctx, monkeypatch):
    """Chromosomes that reach up to 2^32 - 1: where the linearised search keys of the bucketed pass do not fit 32 bits the
    launcher stays on the direct pass; where they fit (one such chromosome) clamped and wrapping keys resolve like the
    oracle's (bits.rs:337-344)."""
    rng = np.random.default_rng(77)
    for n_chroms, expect_bucketed in ((3, False), (1, True)):
        n = 4000
        chr_ = np.sort(rng.integers(0, n_chroms, n))
        offs = np.searchsorted(chr_, np.arange(n_chroms + 1)).astype(np.uint64)
        top = 0xFFFFFFFF if n_chroms > 1 else 0xFF000000  # one chromosome: its LUT bins (+ sentinel) still fit below 2^32
        s = rng.integers(0, top - 0xFFFFF, n)
        e = np.minimum(s + rng.integers(1, 1 << 24, n), top)
        g, o = _both(ctx, "bits", offs, s.astype(np.uint32), e.astype(np.uint32))
        nq = 9001
        qc = rng.integers(0, n_chroms + 1, nq).astype(np.uint32)
        qs = rng.integers(0, 0xFFFFFFFF, nq, dtype=np.uint64)
        qe = np.minimum(qs + rng.integers(1, 1 << 26, nq).astype(np.uint64), 0xFFFFFFFF)
        qs[:50] = 0xFFFFFFFF  # start + 1 wraps
        qe[50:100] = 0xFFFFFFFF
        qs, qe = qs.astype(np.uint32), qe.astype(np.uint32)
        monkeypatch.setenv("GTGPU_COUNT_PARTITION", "1")
        n0 = ctx.launch_count()
        cnt, raw = g.count(qc, qs, qe), g.bits_count(qc, qs, qe)
        assert ctx.launch_count() - n0 == (6 if expect_bucketed else 2)
        monkeypatch.delenv("GTGPU_COUNT_PARTITION")
        assert np.array_equal(cnt, o.count(qc, qs, qe)) and np.array_equal(raw, o.bits_count(qc, qs, qe))


@pytest.mark.parametrize("kind", ["bits", "ailist"])
def test_tokenize_files_unk_rule_and_ragged(ctx, kind):
    rng = np.random.default_rng(11)
    n_chroms = 4
    offs, s, e, v = _random_index(rng, n_chroms, 3000, "overlap")
    g, o = _both(ctx, kind, offs, s, e, v)
    # ragged files: empty files, files with only misses (→ [unk]), files crossing tile boundaries
    sizes = [0, 3, 0, 1500, 1, 0, 700, 2500, 0, 0, 5, 1024, 1023, 1025, 0]
    qc_l, qs_l, qe_l = [], [], []
    for i, k in enumerate(sizes):
        qc, qs, qe = _random_queries(rng, n_chroms, k)
        if i in (1, 4, 10):  # force misses
            qc[:] = 0xFFFFFFFF
        qc_l.append(qc); qs_l.append(qs); qe_l.append(qe)
    qc, qs, qe = np.concatenate(qc_l), np.concatenate(qs_l), np.concatenate(qe_l)
    fo = np.concatenate([[0], np.cumsum(sizes)]).astype(np.uint64)
    unk = 3000
    g_off, g_ids = g.tokenize_files(fo, qc, qs, qe, unk)
    o_off, o_ids = o.tokenize_files(fo, qc, qs, qe, unk)
    assert np.array_equal(g_off, o_off)
    assert np.array_equal(g_ids, o_ids)
    assert (g_ids == unk).sum() >= 8  # the empty and all-miss files
    # no files at all / no queries at all
    g_off, g_ids = g.tokenize_files(np.zeros(1, np.uint64), qc[:0], qs[:0], qe[:0], unk)
    assert list(g_off) == [0] and len(g_ids) == 0
    g_off, g_ids = g.tokenize_files(np.zeros(4, np.uint64), qc[:0], qs[:0], qe[:0], unk)
    assert list(g_off) == [0, 1, 2, 3] and list(g_ids) == [unk] * 3


def test_output_capacity_rerun(ctx):
    """Far more hits than the optimistic output capacity (n + n/4 + 1024): the host wrapper must re-run exactly."""
    n = 4000
    offs = np.array([0, n], dtype=np.uint64)
    s = np.arange(n, dtype=np.uint32)
    e = s + 5000
    g, o = _both(ctx, "bits", offs, s, e)
    nq = 300
    qc = np.zeros(nq, np.uint32)
    qs = np.arange(nq, dtype=np.uint32) * 10
    qe = qs + 3000
    _assert_same_find(g, o, qc, qs, qe)
    fo = np.array([0, 100, 300], dtype=np.uint64)
    g_off, g_ids = g.tokenize_files(fo, qc, qs, qe, n)
    o_off, o_ids = o.tokenize_files(fo, qc, qs, qe, n)
    assert np.array_equal(g_off, o_off) and np.array_equal(g_ids, o_ids)


@pytest.mark.parametrize("kind,nested", [("bits", 0.0), ("ailist", 0.0), ("bits", 0.01), ("ailist", 0.01)])
def test_synthetic_c2_shape_vs_oracle(ctx, kind, nested):
    """The bench workload at 1/1000 scale: 100 k-region hg38 universe (optionally the nested C2n variant),
    40 sorted files x 5 000 regions, 0.1 % unknown chromosomes."""
    from gtars_b200 import synth
    u = synth.make_universe(100_000, nested_frac=nested)
    q = synth.make_query_files(u, 40, 5000, unknown_frac_ppm=1000)
    offs = u["chrom_offsets"].numpy().astype(np.uint64)
    s, e, v = (u[k].numpy().view(np.uint32) for k in ("g_start", "g_end", "g_val"))
    g, o = _both(ctx, kind, offs, s, e, v)
    qc, qs, qe = (q[k].numpy().view(np.uint32) for k in ("chr", "start", "end"))
    fo = q["file_offsets"].numpy().astype(np.uint64)
    g_off, g_ids = g.tokenize_files(fo, qc, qs, qe, u["unk_id"])
    o_off, o_ids = o.tokenize_files(fo, qc, qs, qe, u["unk_id"])
    assert np.array_equal(g_off, o_off)
    assert np.array_equal(g_ids, o_ids)
    assert np.array_equal(g.count(qc, qs, qe), o.count(qc, qs, qe))
    if nested and kind == "ailist":
        assert g.info()["max_components"] >= 2


# ---- IGD / LOLA count matrices and fragment tokenization vs the oracle --------------------------------------------------
@pytest.mark.parametrize("min_overlap", [1, 2, 40])
def test_igd_random_differential(ctx, min_overlap):
    from gtars_b200 import ffi
    from oracle import oracle as orc
    rng = np.random.default_rng(100 + min_overlap)
    n_chroms, n_files = 4, 37
    sizes = rng.integers(0, 400, n_files)
    sizes[5] = 0
    n = int(sizes.sum())
    fo = np.concatenate([[0], np.cumsum(sizes)]).astype(np.uint64)
    dc = rng.integers(0, n_chroms, n).astype(np.uint32)
    ds = rng.integers(0, 300_000, n).astype(np.uint32)
    de = (ds + rng.integers(-20, 40_000, n).clip(-20, None)).astype(np.int64).clip(0, None).astype(np.uint32)  # some empty / reversed
    wide = rng.random(n) < 0.05
    de = np.where(wide, ds + rng.integers(20_000, 120_000, n), de).astype(np.uint32)  # spans many 16 kb tiles
    g = ffi.Igd(ctx, fo, n_chroms, dc, ds, de)
    o = orc.Igd(fo, dc, ds, de)
    set_sizes = [0, 700, 1, 1300, 0, 450]
    nq = sum(set_sizes)
    so = np.concatenate([[0], np.cumsum(set_sizes)]).astype(np.uint64)
    qc = rng.integers(0, n_chroms + 1, nq).astype(np.uint32)
    qc[rng.random(nq) < 0.02] = 0xFFFFFFFF
    qs = rng.integers(0, 320_000, nq).astype(np.uint32)
    qe = (qs + rng.integers(1, 30_000, nq)).astype(np.uint32)
    qe = np.where(rng.random(nq) < 0.05, qs, qe).astype(np.uint32)  # empty queries contribute nothing
    assert np.array_equal(g.count_set_overlaps(so, qc, qs, qe, min_overlap), o.count_set_overlaps(so, qc, qs, qe, min_overlap))
    assert np.array_equal(g.count_region_hits(so, qc, qs, qe, min_overlap), o.count_region_hits(so, qc, qs, qe, min_overlap))
    # single-rank sharded entry point == unsharded
    assert np.array_equal(g.count_sharded(True, n_files, so, qc, qs, qe, min_overlap), o.count_region_hits(so, qc, qs, qe, min_overlap))
    from gtars_b200.ffi import GtarsGpuError
    with pytest.raises(GtarsGpuError):
        g.count_region_hits(so, qc, qs, qe, 0)
    g.close()


@pytest.mark.parametrize("binary", [True, False])
def test_igd_count_dev_any_set_order(ctx, binary):
    """gtgpu_igd_count_dev takes the set of every query as an array: any order is fine (the host entry points pass runs)."""
    import torch
    from gtars_b200 import ffi
    from oracle import oracle as orc
    rng = np.random.default_rng(909 + int(binary))
    n_chroms, n_files, n_sets = 3, 61, 7
    sizes = rng.integers(100, 500, n_files)
    n = int(sizes.sum())
    fo = np.concatenate([[0], np.cumsum(sizes)]).astype(np.uint64)
    dc = rng.integers(0, n_chroms, n).astype(np.uint32)
    ds = rng.integers(0, 1_000_000, n).astype(np.uint32)
    de = (ds + rng.integers(1, 40_000, n)).astype(np.uint32)
    g = ffi.Igd(ctx, fo, n_chroms, dc, ds, de)
    o = orc.Igd(fo, dc, ds, de)
    nq = 23_000
    qc = rng.integers(0, n_chroms + 1, nq).astype(np.uint32)
    qs = rng.integers(0, 1_010_000, nq).astype(np.uint32)
    qe = (qs + rng.integers(1, 30_000, nq)).astype(np.uint32)
    set_of = rng.integers(0, n_sets, nq).astype(np.uint32)            # arbitrary order
    set_of[5000:14000] = 3                                            # ... with one long run across chunk boundaries
    # oracle: group the queries by set (stable), count per set
    order = np.argsort(set_of, kind="stable")
    so = np.concatenate([[0], np.cumsum(np.bincount(set_of, minlength=n_sets))]).astype(np.uint64)
    fn = o.count_region_hits if binary else o.count_set_overlaps
    want = fn(so, qc[order], qs[order], qe[order], 2, threads=orc.max_threads())
    dev = torch.device("cuda", 0)
    t = [torch.from_numpy(a.view(np.int32)).to(dev) for a in (set_of, qc, qs, qe)]
    d_out = torch.zeros(n_sets * n_files, dtype=torch.int64, device=dev)
    ffi.check(ffi.lib().gtgpu_igd_count_dev(g._h, 1 if binary else 0, nq, t[0].data_ptr(), t[1].data_ptr(), t[2].data_ptr(),
                                            t[3].data_ptr(), 2, d_out.data_ptr()))
    ctx.synchronize()
    assert np.array_equal(d_out.cpu().numpy().astype(np.uint64).reshape(n_sets, n_files), want)
    g.close()


@pytest.mark.parametrize("min_overlap", [1, 25])
def test_igd_large_batch_many_sets(ctx, min_overlap):
    """A larger IGD batch (40 k queries, 90 files, 11 query sets incl. empty and one-query sets): both count semantics
    identical to the oracle."""
    from gtars_b200 import ffi
    from oracle import oracle as orc
    rng = np.random.default_rng(555 + min_overlap)
    n_chroms, n_files = 3, 90
    sizes = rng.integers(50, 400, n_files)
    n = int(sizes.sum())
    fo = np.concatenate([[0], np.cumsum(sizes)]).astype(np.uint64)
    dc = rng.integers(0, n_chroms, n).astype(np.uint32)
    ds = rng.integers(0, 2_000_000, n).astype(np.uint32)
    de = (ds + rng.integers(1, 30_000, n)).astype(np.uint32)
    g = ffi.Igd(ctx, fo, n_chroms, dc, ds, de)
    o = orc.Igd(fo, dc, ds, de)
    set_sizes = [5000, 0, 1, 2047, 2048, 2049, 12000, 3, 0, 9000, 7000]
    nq = sum(set_sizes)
    assert nq >= 32768
    so = np.concatenate([[0], np.cumsum(set_sizes)]).astype(np.uint64)
    qc = rng.integers(0, n_chroms + 1, nq).astype(np.uint32)
    qs = rng.integers(0, 2_010_000, nq).astype(np.uint32)
    qe = (qs + rng.integers(1, 20_000, nq)).astype(np.uint32)
    th = orc.max_threads()
    want_pairs = o.count_set_overlaps(so, qc, qs, qe, min_overlap, threads=th)
    want_hits = o.count_region_hits(so, qc, qs, qe, min_overlap, threads=th)
    assert np.array_equal(g.count_set_overlaps(so, qc, qs, qe, min_overlap), want_pairs)
    assert np.array_equal(g.count_region_hits(so, qc, qs, qe, min_overlap), want_hits)
    assert int(want_pairs.sum()) > 100_000
    g.close()


@pytest.mark.parametrize("kind", ["bits", "ailist"])
def test_fragments_random_differential(ctx, kind):
    rng = np.random.default_rng(77)
    n_chroms = 3
    offs, s, e, v = _random_index(rng, n_chroms, 4000, "overlap")
    g, o = _both(ctx, kind, offs, s, e, v)
    n, n_bc = 20_000, 300
    qc, qs, qe = _random_queries(rng, n_chroms, n)
    bc = (rng.zipf(1.5, n) % n_bc).astype(np.uint32)
    bc[bc == 7] = 8  # barcode 7 never appears: empty list
    unk = 4000
    g_off, g_ids = g.tokenize_fragments(qc, qs, qe, bc, n_bc, unk)
    o_off, o_ids = o.tokenize_fragments(qc, qs, qe, bc, n_bc, unk)
    assert np.array_equal(g_off, o_off)
    assert np.array_equal(g_ids, o_ids)
    assert g_off[7] == g_off[8]
    g_off, g_ids = g.tokenize_fragments(qc[:0], qs[:0], qe[:0], bc[:0], 5, unk)
    assert list(g_off) == [0] * 6 and len(g_ids) == 0


@pytest.mark.parametrize("kind", ["bits", "ailist"])
@pytest.mark.parametrize("style,n_bc", [("peaks", 70_000), ("nested", 513), ("overlap", 40)])
def test_fragments_device_resident_entry_point(ctx, kind, style, n_bc):
    """gtgpu_tokenize_fragments_dev (no host copies, no synchronisation) and the host entry point against the oracle:
    lean universes, multi-hit universes (pool lists / generic walk under the per-query [unk] rule), barcode counts that
    take one 8-bit pair-sort pass (40) and the two-pass packed group-by with 8-bit (513) and 9-bit (70 000) low digits,
    degenerate and unknown-chromosome fragments, a partial last tile.  Three and more passes: test_gpu_sort.py."""
    import torch
    rng = np.random.default_rng(zlib.crc32(f"fragdev/{kind}/{style}".encode()))
    n_chroms = 4
    offs, s, e, v = _random_index(rng, n_chroms, 5000, style)
    g, o = _both(ctx, kind, offs, s, e, v)
    n = 150_001
    qc, qs, qe = _random_queries(rng, n_chroms, n, degenerate=True)
    bc = (rng.integers(0, n_bc, n) ** 2 // n_bc).astype(np.uint32)
    unk = 5000
    o_off, o_ids = o.tokenize_fragments(qc, qs, qe, bc, n_bc, unk)
    h_off, h_ids = g.tokenize_fragments(qc, qs, qe, bc, n_bc, unk)
    assert np.array_equal(h_off, o_off) and np.array_equal(h_ids, o_ids)
    dev = torch.device("cuda", 0)
    t = [torch.from_numpy(a.view(np.int32)).to(dev) for a in (qc, qs, qe, bc)]
    cap = int(o_off[-1]) + 17
    d_ids = torch.zeros(cap, dtype=torch.int32, device=dev)
    d_bco = torch.zeros(n_bc + 1, dtype=torch.int64, device=dev)
    d_total = torch.zeros(1, dtype=torch.int64, device=dev)
    g.tokenize_fragments_dev(n, t[0].data_ptr(), t[1].data_ptr(), t[2].data_ptr(), t[3].data_ptr(), n_bc, unk, d_bco.data_ptr(),
                             d_ids.data_ptr(), cap, d_total.data_ptr())
    ctx.synchronize()
    assert int(d_total.item()) == int(o_off[-1])
    assert np.array_equal(d_bco.cpu().numpy().astype(np.uint64), o_off)
    assert np.array_equal(d_ids[:int(o_off[-1])].cpu().numpy().view(np.uint32), o_ids)
    assert np.array_equal(t[3].cpu().numpy().view(np.uint32), bc)      # the caller's barcode array is not modified
    # a buffer that cannot hold the tokens is reported, not overrun
    small = n + 3
    if int(o_off[-1]) > small:
        d_small = torch.zeros(small + 8, dtype=torch.int32, device=dev)
        g.tokenize_fragments_dev(n, t[0].data_ptr(), t[1].data_ptr(), t[2].data_ptr(), t[3].data_ptr(), n_bc, unk, d_bco.data_ptr(),
                                 d_small.data_ptr(), small, d_total.data_ptr())
        ctx.synchronize()
        assert int(d_total.item()) == -1 and int(d_small[small:].abs().sum().item()) == 0


@pytest.mark.parametrize("kind", ["bits", "ailist"])
def test_tokenize_files_pipelined_chunks(ctx, kind, monkeypatch):
    """The chunked H2D / kernel / D2H pipeline of gtgpu_tokenize_files (forced here with 4 096-query chunks) is
    bit-identical to the single-launch path, with file boundaries on, before and after chunk boundaries."""
    rng = np.random.default_rng(321)
    n_chroms = 4
    offs, s, e, v = _random_index(rng, n_chroms, 5000, "overlap")
    g, o = _both(ctx, kind, offs, s, e, v)
    sizes = [4096, 1, 4095, 8192, 3000, 5192, 10, 12278, 4096 * 3, 777]
    qc, qs, qe = _random_queries(rng, n_chroms, sum(sizes))
    qc[:] = qc % n_chroms  # every file has hits: the pipelined path is taken end to end
    fo = np.concatenate([[0], np.cumsum(sizes)]).astype(np.uint64)
    want_off, want_ids = o.tokenize_files(fo, qc, qs, qe, 5000)
    monkeypatch.setenv("GTGPU_PIPE_CHUNK", "4096")
    got_off, got_ids = g.tokenize_files(fo, qc, qs, qe, 5000)
    assert np.array_equal(got_off, want_off) and np.array_equal(got_ids, want_ids)
    # an empty file forces the [unk] fallback: still exact
    sizes2 = sizes[:3] + [0] + sizes[3:]
    fo2 = np.concatenate([[0], np.cumsum(sizes2)]).astype(np.uint64)
    got_off, got_ids = g.tokenize_files(fo2, qc, qs, qe, 5000)
    want_off, want_ids = o.tokenize_files(fo2, qc, qs, qe, 5000)
    assert np.array_equal(got_off, want_off) and np.array_equal(got_ids, want_ids)
    # far more hits than the optimistic capacity: overflow fallback
    monkeypatch.setenv("GTGPU_PIPE_CHUNK", "1024")
    n = 3000
    g2, o2 = _both(ctx, kind, np.array([0, n], dtype=np.uint64), np.arange(n, dtype=np.uint32), np.arange(n, dtype=np.uint32) + 4000)
    q = 5000
    c0, s0 = np.zeros(q, np.uint32), (np.arange(q) % 2500).astype(np.uint32)
    fo3 = np.array([0, 2000, q], dtype=np.uint64)
    a = g2.tokenize_files(fo3, c0, s0, s0 + 300, n)
    b = o2.tokenize_files(fo3, c0, s0, s0 + 300, n)
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])


def test_tokenize_files_runs_variant(ctx, monkeypatch):
    """gtgpu_tokenize_files_runs (chromosome ids as runs) == gtgpu_tokenize_files, on the plain and the chunked path."""
    from gtars_b200 import synth
    u = synth.make_universe(60_000)
    q = synth.make_query_files(u, 12, 3000, unknown_frac_ppm=2000)
    offs = u["chrom_offsets"].numpy().astype(np.uint64)
    s, e, v = (u[k].numpy().view(np.uint32) for k in ("g_start", "g_end", "g_val"))
    g, o = _both(ctx, "bits", offs, s, e, v)
    qc, qs, qe = (q[k].numpy().view(np.uint32) for k in ("chr", "start", "end"))
    fo = q["file_offsets"].numpy().astype(np.uint64)
    # runs: boundaries where the chromosome changes or a file starts
    brk = np.flatnonzero(np.diff(qc.astype(np.int64)) != 0) + 1
    starts = np.unique(np.concatenate([[0], brk, fo[:-1].astype(np.int64)]))
    run_offsets = np.concatenate([starts, [len(qc)]]).astype(np.uint64)
    run_chr = qc[starts]
    want = o.tokenize_files(fo, qc, qs, qe, u["unk_id"])
    for chunk in (None, "4096"):
        if chunk:
            monkeypatch.setenv("GTGPU_PIPE_CHUNK", chunk)
        got = g.tokenize_files_runs(fo, run_offsets, run_chr, qs, qe, u["unk_id"])
        assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1])
    from gtars_b200.ffi import GtarsGpuError
    with pytest.raises(GtarsGpuError):
        g.tokenize_files_runs(fo, run_offsets[:-1], run_chr[:-1], qs, qe, u["unk_id"])  # runs do not cover the queries
    # compact wire format: ends as 16-bit widths + an exception list (wide and reversed regions)
    rng = np.random.default_rng(9)
    qe2 = qe.copy()
    wide = rng.choice(len(qs), 300, replace=False)
    qe2[wide[:200]] = qs[wide[:200]] + rng.integers(65535, 3_000_000, 200).astype(np.uint32)   # too wide for 16 bits
    qe2[wide[200:]] = np.maximum(qs[wide[200:]].astype(np.int64) - rng.integers(0, 500, 100), 0).astype(np.uint32)  # end <= start
    width = qe2.astype(np.int64) - qs.astype(np.int64)
    exc = np.flatnonzero((width < 0) | (width > 65534))
    w16 = np.where((width < 0) | (width > 65534), 0xFFFF, width).astype(np.uint16)
    want2 = o.tokenize_files(fo, qc, qs, qe2, u["unk_id"])
    assert not np.array_equal(want2[1], want[1])
    for chunk in ("1000000000", "4096"):
        monkeypatch.setenv("GTGPU_PIPE_CHUNK", chunk)
        got = g.tokenize_files_compact(fo, run_offsets, run_chr, qs, w16, exc.astype(np.uint64), qe2[exc], u["unk_id"])
        assert np.array_equal(got[0], want2[0]) and np.array_equal(got[1], want2[1])
    got = g.tokenize_files_compact(fo, run_offsets, run_chr, qs, (qe - qs).astype(np.uint16), [], [], u["unk_id"])
    assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1])
    with pytest.raises(GtarsGpuError):
        g.tokenize_files_compact(fo, run_offsets, run_chr, qs, w16, [5, 5], [1, 2], u["unk_id"])  # not strictly increasing
    # packed wire format: one word per query (offset from the block anchor | width), exceptions with absolute coordinates
    from gtars_b200 import ffi
    for wb in (0, 8, 16):
        ro, rc, wbits, pk, an, xi, xs, xe = ffi.marshal_packed(qc, qs, qe2, fo, width_bits=wb)
        assert len(xi) >= 300 and (wb == 0 or wbits == wb)
        for chunk in ("1000000000", "4096"):
            monkeypatch.setenv("GTGPU_PIPE_CHUNK", chunk)
            got = g.tokenize_files_packed(fo, ro, rc, wbits, pk, an, xi, xs, xe, u["unk_id"])
            assert np.array_equal(got[0], want2[0]) and np.array_equal(got[1], want2[1])
    with pytest.raises(GtarsGpuError):
        g.tokenize_files_packed(fo, ro, rc, 0, pk, an, xi, xs, xe, u["unk_id"])  # width_bits out of range
    with pytest.raises(GtarsGpuError):
        g.tokenize_files_packed(fo, ro, rc, wbits, pk, an, [5, 5], [1, 2], [3, 4], u["unk_id"])  # not strictly increasing


@pytest.mark.parametrize("kind", ["bits", "ailist"])
@pytest.mark.parametrize("wide_frac", [0.1, 0.3])
def test_pooled_windows_differential(ctx, kind, wide_frac):
    """Moderately (most windows hold 3-7 candidates) and heavily (8-15, some beyond) overlapping / nested universes and
    narrow queries: the pooled candidate lists of the window table (not the direct runs, rarely the generic walk)
    resolve them; counts above 7 per query also exercise the unpacked-offset warps."""
    rng = np.random.default_rng(4242)
    n = 6000
    chr_ = np.sort(rng.integers(0, 2, n))
    offs = np.concatenate([[0], np.cumsum(np.bincount(chr_, minlength=2))]).astype(np.uint64)
    s = rng.integers(0, 1_500_000, n).astype(np.uint32)
    w = np.where(rng.random(n) < wide_frac, rng.integers(3000, 20000, n), rng.integers(50, 1500, n))
    e = (s + w).astype(np.uint32)
    v = rng.permutation(n).astype(np.uint32)
    g, o = _both(ctx, kind, offs, s, e, v)
    info = g.info()
    assert info["bt_pool_windows"] > 1000
    nq = 20000
    qc = rng.integers(0, 2, nq).astype(np.uint32)
    qs = rng.integers(0, 1_520_000, nq).astype(np.uint32)
    qe = (qs + rng.integers(1, 1 << max(int(info["bt_shift"]), 1), nq)).astype(np.uint32)
    for m in (0, 2, 30):
        _assert_same_find(g, o, qc, qs, qe, m)
    fo = np.array([0, 5000, 5000, 12000, nq], dtype=np.uint64)
    a, b = g.tokenize_files(fo, qc, qs, qe, n), o.tokenize_files(fo, qc, qs, qe, n)
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])


@pytest.mark.parametrize("kind", ["bits", "ailist"])
@pytest.mark.parametrize("nested", [0.0, 0.01])
def test_wide_queries_multi_window(ctx, kind, nested):
    """Queries wider than one bin walk several two-bin windows of the table (up to 8), beyond that the generic path;
    hits must come out once, in the backend's order, whatever mix of direct / pooled / overflow windows they cross."""
    from gtars_b200 import synth
    u = synth.make_universe(200_000, nested_frac=nested)
    offs = u["chrom_offsets"].numpy().astype(np.uint64)
    s, e, v = (u[k].numpy().view(np.uint32) for k in ("g_start", "g_end", "g_val"))
    g, o = _both(ctx, kind, offs, s, e, v)
    sh = int(g.info()["bt_shift"])
    rng = np.random.default_rng(99)
    nq = 30_000
    base = synth.make_query_files(u, 1, nq, sort_files=False, unknown_frac_ppm=1000)
    qc, qs = base["chr"].numpy().view(np.uint32), base["start"].numpy().view(np.uint32)
    width = np.where(rng.random(nq) < 0.9, rng.integers(1, 15 << sh, nq), rng.integers(15 << sh, 60 << sh, nq))
    qe = (qs.astype(np.int64) + width).astype(np.uint32)
    for m in (0, 3, 700):
        _assert_same_find(g, o, qc, qs, qe, m)
    fo = np.array([0, 10_000, nq], dtype=np.uint64)
    a, b = g.tokenize_files(fo, qc, qs, qe, u["unk_id"]), o.tokenize_files(fo, qc, qs, qe, u["unk_id"])
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])


# ---- gtars-scoring: count matrices (SURVEY §8f f2) ---------------------------------------------------------------------------
@pytest.mark.parametrize("style", ["peaks", "overlap"])
def test_score_matrix_vs_oracle(ctx, style):
    from gtars_b200 import ffi
    from oracle import oracle as orc
    rng = np.random.default_rng(zlib.crc32(f"score-{style}".encode()))
    n_chroms, n = 5, 6000
    offs, s, e, v = _random_index(rng, n_chroms, n, style)
    g, o = _both(ctx, "bits", offs, s, e, v)
    sizes = [0, 4000, 1, 0, 9000, 2500, 0]
    nf = sum(sizes)
    fc, fs, fe = _random_queries(rng, n_chroms, nf)
    fe = np.maximum(fe, fs + 6).astype(np.uint32)
    fo = np.concatenate([[0], np.cumsum(sizes)]).astype(np.uint64)
    for mode in (ffi.SCORE_ATAC, ffi.SCORE_CHIP):
        got = g.score_matrix(fo, fc, fs, fe, mode, n)
        want = orc.score_matrix(o, fo, fc, fs, fe, mode, n)
        assert got.dtype == np.uint32 and got.shape == (len(sizes), n)
        assert np.array_equal(got, want), mode
        assert int(got.sum()) > 0
    # fewer columns than vals: out-of-range peaks are dropped exactly like CountMatrix::increment
    got = g.score_matrix(fo, fc, fs, fe, ffi.SCORE_CHIP, n // 2)
    assert np.array_equal(got, orc.score_matrix(o, fo, fc, fs, fe, orc.SCORE_CHIP, n // 2))
    # fragments shorter than the shifts wrap in u32 like the reference's release build: still identical
    fe2 = (fs + rng.integers(0, 12, nf)).astype(np.uint32)
    assert np.array_equal(g.score_matrix(fo, fc, fs, fe2, ffi.SCORE_ATAC, n), orc.score_matrix(o, fo, fc, fs, fe2, orc.SCORE_ATAC, n))
    # no fragments at all
    z = np.zeros(3, np.uint64)
    assert g.score_matrix(z, fc[:0], fs[:0], fe[:0], ffi.SCORE_ATAC, n).sum() == 0


def test_score_barcodes_vs_oracle(ctx):
    from oracle import oracle as orc
    rng = np.random.default_rng(77)
    n_chroms, n = 4, 5000
    offs, s, e, v = _random_index(rng, n_chroms, n, "overlap")
    g, o = _both(ctx, "bits", offs, s, e, v)
    nf, n_bc = 30_000, 700
    fc, fs, fe = _random_queries(rng, n_chroms, nf)
    bc = (rng.integers(0, n_bc, nf) ** 2 // n_bc).astype(np.uint32)  # skewed, some barcodes empty
    g_off, g_pk, g_ct = g.score_barcodes(fc, fs, fe, bc, n_bc)
    o_off, o_pk, o_ct = orc.score_barcodes(o, fc, fs, fe, bc, n_bc)
    assert np.array_equal(g_off, o_off)
    assert np.array_equal(g_pk, o_pk)
    assert np.array_equal(g_ct, o_ct)
    assert int(g_ct.sum()) == int(o.count(fc, fs, fe).sum())
    # empty input / input without a single hit
    off, pk, ct = g.score_barcodes(fc[:0], fs[:0], fe[:0], bc[:0], 5)
    assert list(off) == [0] * 6 and len(pk) == 0 and len(ct) == 0
    none = np.full(10, 0xFFFFFFFF, np.uint32)
    off, pk, ct = g.score_barcodes(none, fs[:10], fe[:10], bc[:10] % 5, 5)
    assert list(off) == [0] * 6 and len(pk) == 0


def test_lean_kernel_and_on_device_fallback(ctx):
    """A universe whose windows are all plain records is served by the lean kernel with the full kernel queued behind it
    as an on-device fallback: narrow queries never need it, a batch with wide / degenerate queries is redone by it within
    the same stream sequence (results identical), and the index then stops trying the lean kernel."""
    from gtars_b200 import synth
    u = synth.make_universe(50_000)
    offs = u["chrom_offsets"].numpy().astype(np.uint64)
    s, e, v = (u[k].numpy().view(np.uint32) for k in ("g_start", "g_end", "g_val"))
    g, o = _both(ctx, "bits", offs, s, e, v)
    info = g.info()
    assert info["bt_pool_windows"] == 0 and info["bt_overflow_bins"] == 0
    q = synth.make_query_files(u, 6, 5000)
    qc, qs, qe = (q[k].numpy().view(np.uint32) for k in ("chr", "start", "end"))
    fo = q["file_offsets"].numpy().astype(np.uint64)

    want = o.tokenize_files(fo, qc, qs, qe, u["unk_id"])
    assert info["lean_kernel"] and not info["lean_fell_back"]
    got = g.tokenize_files(fo, qc, qs, qe, u["unk_id"])
    assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1])
    ctx.synchronize()
    assert not g.info()["lean_fell_back"]                   # narrow queries: the records resolved everything
    # wide and reversed queries: the lean kernel cannot resolve them, its fallback does
    qe_w = qe.copy()
    qe_w[::7] = qs[::7] + 50_000
    qe_w[3::11] = qs[3::11] - np.minimum(qs[3::11], 3)
    want_w = o.tokenize_files(fo, qc, qs, qe_w, u["unk_id"])
    got_w = g.tokenize_files(fo, qc, qs, qe_w, u["unk_id"])
    assert np.array_equal(got_w[0], want_w[0]) and np.array_equal(got_w[1], want_w[1])
    ctx.synchronize()
    assert g.info()["lean_fell_back"]                       # ... and the index remembers
    _assert_same_find(g, o, qc, qs, qe_w)
    got2 = g.tokenize_files(fo, qc, qs, qe, u["unk_id"])    # full kernel only from here on: still exact
    assert np.array_equal(got2[0], want[0]) and np.array_equal(got2[1], want[1])
    # a nested universe never uses the lean kernel
    un = synth.make_universe(20_000, nested_frac=0.02)
    gn = _both(ctx, "bits", un["chrom_offsets"].numpy().astype(np.uint64), *(un[k].numpy().view(np.uint32) for k in ("g_start", "g_end", "g_val")))[0]
    assert not gn.info()["lean_kernel"]
