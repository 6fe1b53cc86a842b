"""MultiChromOverlapper / IndexedRegionSet over a batch of BED files resolved in one device pass (gtgpu_overlaps_bed_files / _gz):
count, any, find and subset_by of every file equal the existing methods on RegionSet(path) and the oracle, position by position
in RegionSet::try_from's order (names the index lacks sorted by their bytes among the others), for Bits and AIList, every
min_overlap, plain / gzip / BGZF / mixed paths, any window size, and on both sides of the subset reduction's 32-bit fold."""
import json
import os

import numpy as np
import pytest

from tests.test_gpu_igd_bed import FORMS, bed_text, edge_texts, write_files
from tests.test_gpu_tokenize_bed_files import c2_batch, file_sorted, local_texts, shuffled_within_files

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MS = (None, 1, 5, 6)


@pytest.fixture(scope="module")
def api():
    from gtars_b200 import api as a
    a.device(0)
    return a


def source_regions(seed=3, n=400):
    """an overlapper source over some of the query files' names (and one they never use): nested and identical regions"""
    rng = np.random.default_rng(seed)
    names = ["chr1", "chr2", "chrX", "chr10", "chr1_random", "chrM", "scaf3", "chrSourceOnly"]
    regs = []
    for _ in range(n):
        s = int(rng.integers(0, 3000))
        regs.append((names[int(rng.integers(0, len(names)))], s, s + int(rng.integers(1, 600))))
    regs += regs[:25]                                                    # identical coordinates: subset_by keys them once
    regs += [(c, s + 10, e - 5) for c, s, e in regs[:40] if e - s > 20]  # nested
    return regs


def hits_of(off, vals):
    return [vals[int(off[i]):int(off[i + 1])].tolist() for i in range(len(off) - 1)]


def regions(rs):
    return [(r.chr, r.start, r.end) for r in rs]


def oracle_results(src, paths, kind, m):
    """the oracle's count / any / find over every file's RegionSet::try_from order, split per file"""
    from oracle import oracle as orc
    names = list(dict.fromkeys(c for c, _, _ in src))
    order = sorted(range(len(src)), key=lambda i: names.index(src[i][0]))  # chromosome-grouped, insertion order kept
    co = np.searchsorted([names.index(src[i][0]) for i in order], np.arange(len(names) + 1)).astype(np.uint64)
    ix = orc.Index(kind, co, [src[i][1] for i in order], [src[i][2] for i in order], order)
    sets = [orc.regionset_from_file(p) for p in paths]
    ids = {n: i for i, n in enumerate(names)}
    q = [r for rs in sets for r in rs]
    c = np.array([ids.get(r[0], 0xFFFFFFFF) for r in q], dtype=np.uint32)
    s, e = np.array([r[1] for r in q], dtype=np.uint32), np.array([r[2] for r in q], dtype=np.uint32)
    mm = m or 0
    fq = np.cumsum([0] + [len(rs) for rs in sets])
    off, vals = ix.find(c, s, e, mm)
    return fq, ix.count(c, s, e, mm), ix.any(c, s, e, mm), hits_of(off, vals)


def same_as_existing(api, src, paths, sample=None, oracle=True):
    """every *_bed_files method == the existing method on RegionSet(paths[f]) (on `sample` files) and == the oracle (all files)"""
    rsets = {f: api.RegionSet(paths[f]) for f in (range(len(paths)) if sample is None else sample)}
    for kind in (api.BITS, api.AILIST):
        mco, irs = api.MultiChromOverlapper(src, kind), api.IndexedRegionSet(src, kind)
        for m in MS:
            cnt, anys = mco.count_overlaps_bed_files(paths, m), mco.any_overlaps_bed_files(paths, m)
            fnd, sub = mco.find_overlaps_bed_files(paths, m), mco.subset_by_bed_files(paths, m)
            ifnd, isub = irs.find_overlaps_bed_files(paths, m), irs.subset_by_overlaps_bed_files(paths, m)
            assert len(cnt) == len(anys) == len(fnd) == len(sub) == len(ifnd) == len(isub) == len(paths)
            for f, rs in rsets.items():
                assert cnt[f].dtype == np.uint32 and anys[f].dtype == bool
                assert cnt[f].tolist() == mco.count_overlaps(rs, m), (paths[f], kind, m)
                assert anys[f].tolist() == mco.any_overlaps(rs, m), (paths[f], kind, m)
                assert hits_of(*fnd[f]) == mco.find_overlaps(rs, m), (paths[f], kind, m)
                assert regions(sub[f]) == regions(mco.subset_by(rs, m)), (paths[f], kind, m)
                assert hits_of(*ifnd[f]) == irs.find_overlaps(rs, m), (paths[f], kind, m)
                assert regions(isub[f]) == regions(irs.subset_by_overlaps(rs, m)), (paths[f], kind, m)
            if oracle:
                fq, oc, oa, of = oracle_results(src, paths, kind, m)
                assert np.array_equal(np.concatenate(cnt), oc) and np.array_equal(np.concatenate(anys), oa), (kind, m)
                assert [h for x in fnd for h in hits_of(*x)] == of, (kind, m)
                assert [len(x) for x in cnt] == np.diff(fq).tolist()


def test_reference_vectors(api, tmp_path):
    """K4 (multi_chrom_overlapper.rs), K11 (test_regionset.py:37-55) and K12 (indexed_region_set.rs) queries as BED files, plain
    and .gz: the golden counts, flags, hits and intersect_all / subset_by regions, after the RegionSet sort."""
    kats = json.load(open(os.path.join(ROOT, "tests", "golden", "kats.json")))
    cases = list(kats["K4_mco"])
    cases += [dict(c, source=c["reference"], min_overlap=None) for c in kats["K12_indexed_region_set"]["cases"]]
    seen = 0
    for i, c in enumerate(cases):
        if not c["query"]:
            continue  # a file without a region line is an error, not an empty query
        text = "".join(f"{q[0]}\t{q[1]}\t{q[2]}\n" for q in c["query"]).encode()
        for form in ("plain", "gzip"):
            paths = write_files(tmp_path, f"k{i}", [text, text], form)
            src = [tuple(r) for r in c["source"]]
            order = sorted(range(len(c["query"])), key=lambda k: (c["query"][k][0].encode(), c["query"][k][1]))
            for kind in (api.BITS, api.AILIST):
                mco, irs = api.MultiChromOverlapper(src, kind), api.IndexedRegionSet(src, kind)
                m = c["min_overlap"]
                if "count" in c:
                    assert [x.tolist() for x in mco.count_overlaps_bed_files(paths, m)] == [[c["count"][k] for k in order]] * 2
                if "any" in c:
                    assert [x.tolist() for x in mco.any_overlaps_bed_files(paths, m)] == [[c["any"][k] for k in order]] * 2
                # the golden hits are sets per query (AIList emits them in its own order), as test_oracle_golden compares them
                if "find" in c and c["find"] and isinstance(c["find"][0], list) and c["find"][0] and isinstance(c["find"][0][0], list):
                    got = [[sorted(list(src[v][1:]) for v in h) for h in hits_of(*x)] for x in mco.find_overlaps_bed_files(paths, m)]
                    assert got == [[sorted(c["find"][k]) for k in order]] * 2
                elif "find" in c:
                    assert [hits_of(*x) for x in irs.find_overlaps_bed_files(paths, m)] == [[c["find"][k] for k in order]] * 2
                if "find_idx" in c:
                    got = [[sorted(h) for h in hits_of(*x)] for x in mco.find_overlaps_bed_files(paths, m)]
                    assert got == [[c["find_idx"][k] for k in order]] * 2
                if "intersect_all" in c:
                    want = [tuple(r) for r in c["intersect_all"]]
                    assert [regions(x) for x in irs.subset_by_overlaps_bed_files(paths)] == [want] * 2
                    assert [regions(x) for x in mco.subset_by_bed_files(paths)] == [sorted(set(want))] * 2
            seen += 1
    assert seen >= 2 * 16


@pytest.mark.parametrize("form", FORMS)
@pytest.mark.parametrize("case", sorted({**edge_texts(), **local_texts()}))
def test_edge_files(api, case, form, tmp_path):
    texts = {**edge_texts(), **local_texts()}[case]
    paths = write_files(tmp_path, case, texts, form)
    sample = None if len(paths) <= 16 else list(range(8)) + list(range(len(paths) - 8, len(paths)))
    same_as_existing(api, source_regions(), paths, sample=sample)


def test_unknown_names_in_string_order(api, tmp_path):
    """Names the index lacks (chr1_random, chrA) sort by their bytes between the known ones (chr1 < chr10 < chr1_random < chr2 <
    chrA < chrX), equal starts across names: results line up with RegionSet(path) position by position, which they would not if
    unknown names went last."""
    names = ["chrX", "chrA", "chr2", "chr1_random", "chr10", "chr1"]
    rows = [(n, s) for s in (100, 200, 300) for n in names]
    texts = ["".join(f"{n}\t{s}\t{s + 50}\n" for n, s in rows[k:] + rows[:k]).encode() for k in range(0, len(rows), 5)]
    src = [(n, s - 10, s + 20) for n in ("chr1", "chr10", "chr2", "chrX") for s in (100, 200, 300)]
    for form in ("plain", "gzip"):
        paths = write_files(tmp_path, "unknown", texts, form)
        same_as_existing(api, src, paths)
        counts = api.MultiChromOverlapper(src, api.BITS).count_overlaps_bed_files(paths)
        for c, p in zip(counts, paths):
            rs = list(api.RegionSet(p))
            assert [r.chr for r in rs][:6] == ["chr1", "chr1", "chr1", "chr10", "chr10", "chr10"]
            assert c.tolist() == [0 if r.chr in ("chr1_random", "chrA") else 1 for r in rs]


def test_forced_windows(api, tmp_path, monkeypatch):
    """GTGPU_INGEST_WINDOW of 1 byte to 64 KiB gives the default window's results, plain and BGZF."""
    t = {**edge_texts(), **local_texts()}
    sets = {k: t[k] for k in ("no_final_newline", "comments_crlf", "header_in_file_3", "sorted_and_unsorted", "equal_starts")}
    sets["tiny"] = t["tiny_files"][:300]
    src = source_regions()
    mco = api.MultiChromOverlapper(src, api.AILIST)
    irs = api.IndexedRegionSet(src, api.BITS)

    def run(paths):
        return ([x.tolist() for x in mco.count_overlaps_bed_files(paths, 5)],
                [[hits_of(*x)] for x in mco.find_overlaps_bed_files(paths)],
                [regions(x) for x in mco.subset_by_bed_files(paths)],
                [regions(x) for x in irs.subset_by_overlaps_bed_files(paths)])

    paths = {k: (write_files(tmp_path, k, v, "plain"), write_files(tmp_path, k, v, "bgzf")) for k, v in sets.items()}
    monkeypatch.delenv("GTGPU_INGEST_WINDOW", raising=False)
    want = {k: run(p[0]) for k, p in paths.items()}
    for w in ("1", "7", "64", "1024", "65536"):
        monkeypatch.setenv("GTGPU_INGEST_WINDOW", w)
        for k, (plain, bg) in paths.items():
            assert run(plain) == want[k], (w, k)
            assert run(bg) == want[k], (w, k)


def test_errors_and_no_files(api, tmp_path, monkeypatch):
    """A malformed line names its file and 1-based line (across a forced window boundary too); a file without a region line is
    rejected; the overlapper stays usable after each error; [] gives []."""
    from gtars_b200 import ffi
    rng = np.random.default_rng(9)
    good = [("\n".join(f"chr{1 + j % 2}\t{int(rng.integers(0, 3000))}\t3500" for j in range(300)) + "\n").encode() for _ in range(6)]
    good_paths = write_files(tmp_path, "good", good, "plain")
    src = source_regions()
    mco, irs = api.MultiChromOverlapper(src, api.BITS), api.IndexedRegionSet(src, api.AILIST)
    want = [x.tolist() for x in mco.count_overlaps_bed_files(good_paths)]

    def still_usable():
        assert [x.tolist() for x in mco.count_overlaps_bed_files(good_paths)] == want

    for k, j, window in ((0, 2, None), (3, 17, None), (5, 290, "4096"), (4, 300, "1")):
        if window:
            monkeypatch.setenv("GTGPU_INGEST_WINDOW", window)
        lines = good[k].decode().split("\n")
        lines[j - 1] = "chr1\tabc\t100"
        bad = list(good)
        bad[k] = "\n".join(lines).encode()
        for form in ("plain", "gzip", "mixed"):
            paths = write_files(tmp_path, f"bad{k}", bad, form)
            for call in (mco.count_overlaps_bed_files, mco.subset_by_bed_files, irs.find_overlaps_bed_files):
                with pytest.raises(api.GtarsError) as e:
                    call(paths)
                assert paths[k] in str(e.value) and f"line {j}" in str(e.value), str(e.value)
                still_usable()
        monkeypatch.delenv("GTGPU_INGEST_WINDOW", raising=False)
    for empty in (b"", b"# only\n#comments\ntrack x\n", b"chrom\tstart\tend\n"):
        paths = write_files(tmp_path, "empty", good[:2] + [empty] + good[2:], "plain")
        with pytest.raises(api.GtarsError) as e:
            mco.any_overlaps_bed_files(paths)
        assert paths[2] in str(e.value) and "0 regions" in str(e.value)
        still_usable()
    assert mco.count_overlaps_bed_files([]) == [] and mco.find_overlaps_bed_files([]) == []
    assert mco.subset_by_bed_files([]) == [] and irs.subset_by_overlaps_bed_files([]) == [] and irs.find_overlaps_bed_files([]) == []
    # the raw ABI: zero files give [0] and empty buffers; a keys table must cover every val
    ctx = ffi.Context(0)
    ix = ffi.Index(ctx, ffi.KIND_BITS, np.array([0, 3], dtype=np.uint64), [1, 5, 9], [4, 8, 12], [0, 1, 2])
    for mode in range(4):
        fq, off, vals = ix.overlaps_bed_text(mode, b"", np.zeros(1, dtype=np.uint64), ["chr1"])
        assert fq.tolist() == [0] and len(vals) == 0 and (off is None if mode < 2 else off.tolist() == [0])
        fq, off, vals = ix.overlaps_bed_gz(mode, b"", np.zeros(1, dtype=np.uint64), np.zeros(1, dtype=np.uint64), ["chr1"])
        assert fq.tolist() == [0] and len(vals) == 0
    one = b"chr1\t0\t20\n"
    fo = np.array([0, len(one)], dtype=np.uint64)
    with pytest.raises(ffi.GtarsGpuError) as e:
        ix.overlaps_bed_text(3, one, fo, ["chr1"], keys=[0, 0])
    assert e.value.code == 1 and "keys" in str(e.value)
    fq, off, vals = ix.overlaps_bed_text(3, one, fo, ["chr1"], keys=[7, 3, 7])
    assert fq.tolist() == [0, 1] and off.tolist() == [0, 2] and vals.tolist() == [3, 7]
    ix.close()
    ctx.close()


def _big_source(n, seed):
    rng = np.random.default_rng(seed)
    names = ["chr1", "chr2", "chr3"]
    s = rng.integers(0, 2_000_000, n)
    regs = [(names[i % 3], int(a), int(a) + int(w)) for i, (a, w) in enumerate(zip(s, rng.integers(50, 3000, n)))]
    return regs + regs[: n // 50]


@pytest.mark.parametrize("n_files,n_src", [(40, 5000), (33_000, 70_000)])
def test_subset_on_both_sides_of_the_fold(api, tmp_path, n_files, n_src):
    """bits(n_files - 1) + bits(n_keys) <= 32 (one radix pass over file << key_bits | key) and > 32 (16 + 17 bits: by key, then
    a pass by file): subset_by_bed_files / subset_by_overlaps_bed_files equal the host methods on a sample of files and, on every
    file, the distinct hit keys of the oracle's find."""
    rng = np.random.default_rng(n_files)
    src = _big_source(n_src, 1)
    per = 1 if n_files > 1000 else 200
    texts = []
    for f in range(n_files):
        a = rng.integers(0, 2_000_000, per)
        texts.append("".join(f"chr{1 + int(rng.integers(0, 4))}\t{int(x)}\t{int(x) + int(rng.integers(1, 5000))}\n" for x in a).encode())
    paths = write_files(tmp_path, "fold", texts, "plain")
    sample = list(range(5)) + list(range(n_files - 5, n_files))
    for kind in (api.BITS, api.AILIST):
        mco, irs = api.MultiChromOverlapper(src, kind), api.IndexedRegionSet(src, kind)
        sub, isub = mco.subset_by_bed_files(paths), irs.subset_by_overlaps_bed_files(paths)
        for f in sample:
            rs = api.RegionSet(paths[f])
            assert regions(sub[f]) == regions(mco.subset_by(rs)) and regions(isub[f]) == regions(irs.subset_by_overlaps(rs))
        fq, _, _, of = oracle_results(src, paths, kind, None)
        want = [sorted({v for q in range(fq[f], fq[f + 1]) for v in of[q]}) for f in range(n_files)]
        assert [[src[i] for i in w] for w in want] == [regions(x) for x in isub]
        assert [sorted({src[i] for i in w}) for w in want] == [regions(x) for x in sub]


def test_c2_shape_sorted_and_shuffled():
    """200 files x 50 000 regions (synth, C2-shaped) against a 1e6-peak source as BED text, sorted and shuffled within every
    file: count / any / find equal the existing entry points on the per-file sorted arrays, and the oracle's counts."""
    from gtars_b200 import ffi, synth
    from oracle import oracle as orc
    per = 50_000
    ix_args, (c, s, e), _ = c2_batch(200, per)
    ctx = ffi.Context(0)
    variants = ((c, s, e), shuffled_within_files(c, s, e, per, np.random.default_rng(1)))
    for kind in (ffi.KIND_BITS, ffi.KIND_AILIST):
        ix = ffi.Index(ctx, kind, *ix_args)
        for k, (cc, s2, e2) in enumerate(variants):
            sc, ss, se = file_sorted(cc, s2, e2, per)    # RegionSet::sort of every file (stable: ties keep the file's order)
            want_cnt = ix.count(sc, ss, se, 5)
            want_off, want_vals = ix.find(sc, ss, se)
            if kind == ffi.KIND_BITS and k == 0:
                assert np.array_equal(want_cnt, orc.Index(kind, *ix_args).count(sc, ss, se, 5, threads=0))
            text = bed_text(cc.astype(np.int64), s2, e2)
            fo = np.concatenate([[0], np.flatnonzero(text == 10)[per - 1::per] + 1]).astype(np.uint64)
            fq, _, cnt = ix.overlaps_bed_text(ffi.OVERLAPS_COUNT, text, fo, synth.CHROM_NAMES, 5)
            assert fq.tolist() == list(range(0, 200 * per + 1, per)) and np.array_equal(cnt, want_cnt)
            _, _, anys = ix.overlaps_bed_text(ffi.OVERLAPS_ANY, text, fo, synth.CHROM_NAMES, 5)
            assert np.array_equal(anys.astype(bool), want_cnt > 0)
            _, off, vals = ix.overlaps_bed_text(ffi.OVERLAPS_FIND, text, fo, synth.CHROM_NAMES)
            assert np.array_equal(off, want_off) and np.array_equal(vals, want_vals)
            _, soff, svals = ix.overlaps_bed_text(ffi.OVERLAPS_SUBSET, text, fo, synth.CHROM_NAMES)
            for f in (0, 77, 199):
                a, b = int(want_off[f * per]), int(want_off[(f + 1) * per])
                assert svals[int(soff[f]):int(soff[f + 1])].tolist() == np.unique(want_vals[a:b]).tolist()
            del text
        ix.close()
    ctx.close()


def test_multi_device_context_equals_single():
    """On a context over several devices the call runs on the first one and returns what a single-device context returns."""
    from gtars_b200 import ffi
    if ffi.device_count() < 2:
        pytest.skip("needs at least 2 GPUs")
    texts = local_texts()["sorted_and_unsorted"]
    fo = np.cumsum([0] + [len(t) for t in texts]).astype(np.uint64)
    names = ["chr1", "chr2", "chrX", "chr10"]
    rng = np.random.default_rng(2)
    s = rng.integers(0, 3000, 400).astype(np.uint32)
    args = (np.arange(5, dtype=np.uint64) * 100, s, s + 200, np.arange(400, dtype=np.uint32))
    out = []
    for ctx in (ffi.Context(0), ffi.Context(devices=[0, 1])):
        ix = ffi.Index(ctx, ffi.KIND_AILIST, *args)
        out.append([ix.overlaps_bed_text(m, b"".join(texts), fo, names, 5) for m in range(4)])
        ix.close()
        ctx.close()
    for a, b in zip(*out):
        assert all((x is None and y is None) or np.array_equal(x, y) for x, y in zip(a, b))
