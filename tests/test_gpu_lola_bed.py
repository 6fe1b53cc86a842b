"""Query sets and the LOLA universe from their BED files, parsed on the device (gtgpu_igd_count_bed / _gz, ffi.Igd.count_bed_text /
count_bed_gz, api.Igd.count_bed_files, api.lola_contingency_from_bed_files), count exactly as the same files read by the host
parser (RegionSet(p)) and counted with Igd.count_region_hits / count_set_overlaps / lola_contingency do: plain text, one gzip
member per file, and a mix of plain and .gz paths, in windows of GTGPU_INGEST_WINDOW bytes."""
import gzip
import os
import re

import numpy as np
import pytest

from tests import helpers
from tests.test_gpu_igd_bed import bed_text, edge_texts, synth_db, write_files

pytestmark = pytest.mark.gpu

FORMS = ("plain", "gzip", "mixed")


@pytest.fixture(scope="module")
def api():
    from gtars_b200 import api as a
    a.device(0)
    return a


@pytest.fixture(scope="module")
def ctx():
    from gtars_b200 import ffi
    c = ffi.Context(0)
    yield c
    c.close()


def set_texts(sets):
    return [("".join(f"{c}\t{s}\t{e}\n" for c, s, e in st)).encode() for st in sets]


def same_as_host(api, db, paths, m=1):
    """count_bed_files == count_region_hits / count_set_overlaps of RegionSet(p) for every path (one host-array pass each)"""
    sets = [api.RegionSet(p) for p in paths]
    want_hits, want_pairs = db._count(sets, m, False), db._count(sets, m, True)
    assert np.array_equal(db.count_bed_files(paths, m), want_hits), (paths[:2], m)
    assert np.array_equal(db.count_bed_files(paths, m, pairwise=True), want_pairs), (paths[:2], m)
    return want_hits


def same_lola_as_host(api, db, user_paths, universe_path, m=1):
    got = api.lola_contingency_from_bed_files(db, user_paths, universe_path, m)
    want = api.lola_contingency(db, [api.RegionSet(p) for p in user_paths], api.RegionSet(universe_path), m)
    assert got.dtype == np.int64 and np.array_equal(got, want), (user_paths[:2], universe_path, m)
    return got


@pytest.mark.parametrize("form", FORMS)
def test_lola_kats(api, golden, form, tmp_path):
    """K9: enrichment.rs:830-1104 with database, user sets and universe as BED files (1,1,2,6; binary support; min_overlap 10 /
    11; the negative b that passes through)."""
    for i, case in enumerate(golden[1]["K9_lola"]):
        db = api.Igd.from_bed_files(write_files(tmp_path, f"db{i}", set_texts(case["db"]), form))
        user = write_files(tmp_path, f"user{i}", set_texts(case["user"]), form)
        universe = write_files(tmp_path, f"universe{i}", set_texts([case["universe"]] * 2), form)[1]  # a .gz path in "mixed"
        t = same_lola_as_host(api, db, user, universe, case["min_overlap"])
        if "abcd" in case:
            assert t.tolist() == case["abcd"], case["cite"]
        if "support" in case:
            assert t[:, :, 0].tolist() == case["support"], case["cite"]


@pytest.mark.parametrize("form", FORMS)
def test_reference_fixtures(api, golden, fixture_dir, form, tmp_path):
    """lola_multi_db loaded three ways (Igd([RegionSet]), Igd.from_bed_files, from_igd_file after save); queries query1 / query2
    and every database file: count_bed_files == count_region_hits / count_set_overlaps of RegionSet(p), and the LOLA tables ==
    lola_contingency == the oracle's count_region_hits + lola_tables."""
    from oracle import oracle as orc
    k8 = golden[1]["K8_inputs"]
    texts = [open(os.path.join(fixture_dir, r), "rb").read() for r in k8["dbs"]["lola_multi_db"]]
    db_paths = write_files(tmp_path, "db", texts, form)
    q_texts = [open(os.path.join(fixture_dir, q), "rb").read() for q in k8["queries"]]
    q_paths = write_files(tmp_path, "q", q_texts + texts, form)
    sets = [api.RegionSet(p) for p in db_paths]
    host = api.Igd(sets)
    saved = str(tmp_path / f"lola_{form}.igd")
    host.save(saved)
    cmap = helpers.ChromMap()
    fo, dc, ds, de = helpers.flatten_sets([[(r.chr, r.start, r.end) for r in s] for s in sets], cmap, add=True)
    oracle_db = orc.Igd(fo, dc, ds, de)
    qo, qc, qs, qe = helpers.flatten_sets([[(r.chr, r.start, r.end) for r in api.RegionSet(p)] for p in q_paths], cmap)
    for name, db in (("sets", host), ("bed", api.Igd.from_bed_files(db_paths)), ("igd_file", api.Igd.from_igd_file(saved))):
        for m in (1, 2, 10, 11, 500):
            hits = same_as_host(api, db, q_paths, m)
            assert np.array_equal(hits, oracle_db.count_region_hits(qo, qc, qs, qe, m)), (name, m)
        t = same_lola_as_host(api, db, q_paths[1:], q_paths[0])
        hits = oracle_db.count_region_hits(qo, qc, qs, qe, 1)
        want = orc.lola_tables(hits[1:], hits[0], np.diff(qo)[1:], int(np.diff(qo)[0]))
        assert np.array_equal(t, want), name
        assert t[:, :, 0].sum() > 0


@pytest.mark.parametrize("form", FORMS)
@pytest.mark.parametrize("case", sorted(edge_texts()))
def test_edge_files(api, case, form, tmp_path):
    """header rows, comments, \\r\\n, no final newline, names absent from the database, start >= end and coordinates >= 2^31 (in
    the set sizes, no hits), 1 file and 5 000 files: count_bed_files and the LOLA tables equal the host path."""
    texts = edge_texts()[case]
    if case == "tiny_files" and form in ("gzip", "mixed"):
        texts = texts[:1000]
    rng = np.random.default_rng(2)
    db_sets = [[(n, int(s), int(s) + int(rng.integers(1, 300))) for n, s in
                zip(rng.choice(["chr1", "chr2", "chr10", "chr1_random", "chrM", "chrOnlyInDb"], 400), rng.integers(0, 3200, 400))]
               for _ in range(5)]
    db = api.Igd.from_bed_files(write_files(tmp_path, "db", set_texts(db_sets), "plain"))
    paths = write_files(tmp_path, case, texts, form)
    for m in (1, 7):
        same_as_host(api, db, paths, m)
    same_lola_as_host(api, db, paths[:-1] or paths, paths[-1])


def _file_line(msg):
    m = re.search(r"file (\d+), line (\d+)", msg)
    assert m, msg
    return int(m.group(1)), int(m.group(2))


def test_errors(api, ctx, tmp_path):
    """A malformed line names its path (ffi: file index) and 1-based line; a file without a region line gives "0 regions found"
    with its path; min_overlap = 0 and an Igd from from_single_region_set raise.  The next call succeeds after each."""
    from gtars_b200 import ffi
    rng = np.random.default_rng(9)
    good = [("\n".join(f"chr{1 + j % 2}\t{int(rng.integers(0, 5000))}\t6000" for j in range(300)) + "\n").encode() for _ in range(5)]
    db = api.Igd.from_bed_files(write_files(tmp_path, "db", good[:3], "plain"))
    names = ["chr1", "chr2"]
    g, _ = ffi.Igd.from_bed_text(ctx, b"".join(good[:3]), np.cumsum([0] + [len(t) for t in good[:3]]).astype(np.uint64))
    ok_paths = write_files(tmp_path, "ok", good, "plain")
    want = db.count_bed_files(ok_paths)
    fo = np.cumsum([0] + [len(t) for t in good]).astype(np.uint64)
    want_ffi = g.count_bed_text(True, b"".join(good), fo, names)

    def still_usable():
        assert np.array_equal(db.count_bed_files(ok_paths), want)
        got = g.count_bed_text(True, b"".join(good), fo, names)
        assert np.array_equal(got[0], want_ffi[0]) and np.array_equal(got[1], want_ffi[1])

    for k, j in ((0, 2), (3, 17), (4, 300)):
        lines = good[k].decode().split("\n")
        lines[j - 1] = "chr1\tabc\t100"
        bad = list(good)
        bad[k] = "\n".join(lines).encode()
        for form in FORMS:
            paths = write_files(tmp_path, f"bad{k}", bad, form)
            with pytest.raises(api.GtarsError) as e:
                db.count_bed_files(paths)
            assert paths[k] in str(e.value) and f"line {j}" in str(e.value), str(e.value)
            with pytest.raises(api.GtarsError) as e:
                api.lola_contingency_from_bed_files(db, paths[:-1], paths[-1])
            assert paths[k] in str(e.value), str(e.value)
            still_usable()
        bfo = np.cumsum([0] + [len(t) for t in bad]).astype(np.uint64)
        members = [gzip.compress(t, mtime=0) for t in bad]
        mo = np.cumsum([0] + [len(x) for x in members]).astype(np.uint64)
        for call in (lambda: g.count_bed_text(False, b"".join(bad), bfo, names),
                     lambda: g.count_bed_gz(False, b"".join(members), np.arange(len(bad) + 1), mo, names)):
            with pytest.raises(ffi.GtarsGpuError) as e:
                call()
            assert e.value.code == 1 and _file_line(str(e.value)) == (k, j), str(e.value)
            still_usable()
    for empty in (b"", b"# only\n#comments\ntrack x\n", b"chrom\tstart\tend\n"):
        texts = good[:2] + [empty]
        for form in ("plain", "gzip"):
            paths = write_files(tmp_path, "empty", texts, form)
            with pytest.raises(api.GtarsError) as e:
                db.count_bed_files(paths)
            assert paths[2] in str(e.value) and "0 regions" in str(e.value), str(e.value)
            with pytest.raises(api.GtarsError) as e:        # an empty universe fails in the parse, naming its path
                api.lola_contingency_from_bed_files(db, paths[:2], paths[2])
            assert paths[2] in str(e.value) and "0 regions" in str(e.value), str(e.value)
            still_usable()
    for m in (0, -1):
        with pytest.raises(api.GtarsError):
            db.count_bed_files(ok_paths, m)
        with pytest.raises(api.GtarsError):
            api.lola_contingency_from_bed_files(db, ok_paths[:2], ok_paths[2], m)
        with pytest.raises(ffi.GtarsGpuError) as e:
            g.count_bed_text(True, b"".join(good), fo, names, min_overlap=m)
        assert e.value.code == 6
        still_usable()
    single = api.Igd.from_single_region_set([("chr1", 0, 100)])
    with pytest.raises(api.GtarsError):
        single.count_bed_files(ok_paths)
    with pytest.raises(api.GtarsError):
        api.lola_contingency_from_bed_files(single, ok_paths[:2], ok_paths[2])
    still_usable()
    g.close()


def test_forced_windows(api, ctx, tmp_path, monkeypatch):
    """Windows of 1 byte to 64 KiB give the default window's matrices and set sizes, including set boundaries exactly on
    window cuts (every set of "aligned" is 64 bytes)."""
    from gtars_b200 import ffi
    texts = edge_texts()
    rng = np.random.default_rng(8)
    aligned = []
    for i in range(40):
        s = int(rng.integers(0, 3000))
        line = f"chr{1 + i % 3}\t{s:010d}\t{s + 50:010d}"
        aligned.append((line + "\n" + line[:-1] + "7" + "\t" + "x" * 9 + "\n").encode())
    assert all(len(t) == 64 for t in aligned)
    sets = {"aligned": aligned, "no_final_newline": texts["no_final_newline"], "comments_crlf": texts["comments_crlf"],
            "header_in_file_3": texts["header_in_file_3"], "tiny": texts["tiny_files"][:300]}
    db_sets = [[(f"chr{1 + j % 3}", int(s), int(s) + 200) for j, s in enumerate(rng.integers(0, 3200, 300))] for _ in range(4)]
    db_texts = set_texts(db_sets)
    db = api.Igd.from_bed_files(write_files(tmp_path, "db", db_texts, "plain"))
    g, names = ffi.Igd.from_bed_text(ctx, b"".join(db_texts), np.cumsum([0] + [len(t) for t in db_texts]).astype(np.uint64))
    paths = {k: write_files(tmp_path, k, v, "gzip") + write_files(tmp_path, k, v, "plain") for k, v in sets.items()}
    monkeypatch.delenv("GTGPU_INGEST_WINDOW", raising=False)

    def run(k, v):
        fo = np.cumsum([0] + [len(t) for t in v]).astype(np.uint64)
        mats = [db.count_bed_files(half, 1, pw) for half in (paths[k][:len(v)], paths[k][len(v):]) for pw in (False, True)]
        mats += list(g.count_bed_text(True, b"".join(v), fo, names)) + list(g.count_bed_text(False, b"".join(v), fo, names))
        return mats

    want = {k: run(k, v) for k, v in sets.items()}
    for k, v in sets.items():
        same_as_host(api, db, paths[k][len(v):])
        assert np.array_equal(want[k][5], [len(api.RegionSet(p)) for p in paths[k][len(v):]])
    for w in ("1", "7", "64", "1024", "65536"):
        monkeypatch.setenv("GTGPU_INGEST_WINDOW", w)
        for k, v in sets.items():
            got = run(k, v)
            assert all(np.array_equal(a, b) for a, b in zip(got, want[k])), (w, k)
    g.close()


def _c4_inputs(n_db=2000, per_db=20_000, n_user=200, per_user=10_000, n_universe=1_000_000, seed=31):
    """C4's shape, reduced: database arrays, and the user sets (sampled from the universe) plus the universe as BED texts"""
    c, s, e = synth_db(n_db, per_db, seed)
    rng = np.random.default_rng(seed + 1)
    uc = rng.integers(0, 25, n_universe).astype(np.int64)
    us = rng.integers(0, 2**28, n_universe).astype(np.uint32)
    ue = (us + rng.integers(1, 5000, n_universe)).astype(np.uint32)
    pick = [rng.choice(n_universe, per_user, replace=False) for _ in range(n_user)] + [np.arange(n_universe)]
    texts = [bed_text(uc[p], us[p], ue[p]) for p in pick]
    qc = np.concatenate([uc[p] for p in pick]).astype(np.uint32)
    qs = np.concatenate([us[p] for p in pick])
    qe = np.concatenate([ue[p] for p in pick])
    so = np.cumsum([0] + [len(p) for p in pick]).astype(np.uint64)
    return (c, s, e), texts, (so, qc, qs, qe)


def test_c4_shape_reduced(ctx):
    """2 000 database sets x 2e4 regions; 200 user sets x 1e4 regions sampled from a 1e6-region universe, and the universe:
    as plain text and as gzip members, the matrices equal ffi.Igd.count_region_hits / count_set_overlaps on the same arrays.
    The database names its last chromosome differently from the query files: those queries are unknown names and hit nothing,
    as an unknown id does in the array call."""
    from gtars_b200 import ffi, synth
    (c, s, e), texts, (so, qc, qs, qe) = _c4_inputs()
    db = ffi.Igd(ctx, np.arange(0, len(c) + 1, 20_000, dtype=np.uint64), 25, c, s, e)
    names = list(synth.CHROM_NAMES[:24]) + ["chrM_absent_from_queries"]
    qc_ref = np.where(qc == 24, np.uint32(0xFFFFFFFF), qc).astype(np.uint32)
    want = {True: db.count_region_hits(so, qc_ref, qs, qe), False: db.count_set_overlaps(so, qc_ref, qs, qe)}
    assert want[True].sum() > 0
    text = np.concatenate(texts)
    fo = np.cumsum([0] + [t.nbytes for t in texts]).astype(np.uint64)
    members = [gzip.compress(t.tobytes(), compresslevel=1, mtime=0) for t in texts]
    mo = np.cumsum([0] + [len(m) for m in members]).astype(np.uint64)
    gz = b"".join(members)
    for binary in (True, False):
        for got, regions in (db.count_bed_text(binary, text, fo, names),
                             db.count_bed_gz(binary, gz, np.arange(len(texts) + 1), mo, names)):
            assert np.array_equal(got, want[binary]), binary
            assert np.array_equal(regions, np.diff(so)), binary
    db.close()


def test_multi_device_context_equals_single(ctx):
    """A context over two devices: the parse runs on the first device, every device counts its shard of the database from
    the parsed queries there; matrices and set sizes equal the single device's."""
    from gtars_b200 import ffi, synth
    if ffi.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    (c, s, e), texts, _ = _c4_inputs(n_db=37, per_db=3000, n_user=9, per_user=2000, n_universe=50_000, seed=41)
    fo_db = np.arange(0, len(c) + 1, 3000, dtype=np.uint64)
    names = list(synth.CHROM_NAMES[:24]) + ["chrM_absent_from_queries"]
    text = np.concatenate(texts)
    fo = np.cumsum([0] + [t.nbytes for t in texts]).astype(np.uint64)
    members = [gzip.compress(t.tobytes(), compresslevel=1, mtime=0) for t in texts]
    mo = np.cumsum([0] + [len(m) for m in members]).astype(np.uint64)
    gz = b"".join(members)
    one = ffi.Igd(ctx, fo_db, 25, c, s, e)
    multi = ffi.Context(devices=[0, 1])
    two = ffi.Igd(multi, fo_db, 25, c, s, e)
    for binary in (True, False):
        for m in (1, 9):
            want = one.count_bed_text(binary, text, fo, names, m)
            assert want[0].sum() > 0
            for got in (two.count_bed_text(binary, text, fo, names, m),
                        two.count_bed_gz(binary, gz, np.arange(len(texts) + 1), mo, names, m)):
                assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1]), (binary, m)
    two.close()
    one.close()
    multi.close()
