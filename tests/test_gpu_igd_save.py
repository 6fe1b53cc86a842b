""".igd files written from the device (gtgpu_igd_serialize, ffi.Igd.save_bytes, api.Igd.save) for a database built any way:
from RegionSets, from BED files (plain, gzip, mixed), from an .igd file, or on a multi-device context.  The .igd bytes equal
the host writer's (api.write_igd_file) and the oracle's, and the .tsv equals the host writer's."""
import gzip
import hashlib
import os

import numpy as np
import pytest

from tests.test_gpu_igd_bed import bed_text, synth_db

pytestmark = pytest.mark.gpu

FORMS = ("sets", "plain", "gzip", "mixed")
NBP = 16384


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


def write_texts(d, name, texts, form):
    """texts as BED files; "gzip": one gzip member each; "mixed": alternating plain and .gz paths"""
    paths = []
    for i, t in enumerate(texts):
        gz = form == "gzip" or (form == "mixed" and i % 2 == 1)
        p = str(d / f"{name}_{form}_{i:03d}.bed{'.gz' if gz else ''}")
        with open(p, "wb") as f:
            f.write(gzip.compress(t, mtime=0) if gz else t)
        paths.append(p)
    return paths


def build(api, paths, form):
    return api.Igd([api.RegionSet(p) for p in paths]) if form == "sets" else api.Igd.from_bed_files(paths)


def read(p):
    with open(p, "rb") as f:
        return f.read()


def oracle_bytes(sets, names_of_files, path):
    """orc.Igd over the sets' regions in their order (Igd::from_named_region_sets + save)"""
    from oracle import oracle as orc
    ids, fo, c, s, e = {}, [0], [], [], []
    for rs in sets:
        for r in rs:
            c.append(ids.setdefault(r.chr, len(ids)))
            s.append(r.start)
            e.append(r.end)
        fo.append(len(c))
    orc.Igd(np.array(fo, dtype=np.uint64), c, s, e).save(path, list(ids))
    return read(path)


def same_as_host_writer(api, db, sets, names, d, tag):
    """db.save == api.write_igd_file(sets) == the oracle, .igd and .tsv"""
    got, want = str(d / f"{tag}_dev.igd"), str(d / f"{tag}_host.igd")
    db.save(got, names)
    api.write_igd_file(sets, names, want)
    assert read(got) == read(want), tag
    assert read(got[:-4] + ".tsv") == read(want[:-4] + ".tsv"), tag
    assert read(got) == oracle_bytes(sets, names, str(d / f"{tag}_orc.igd")), tag
    return got


@pytest.mark.parametrize("form", FORMS)
@pytest.mark.parametrize("db", ["lola_multi_db", "igd_file_list_01", "igd_file_list_02"])
def test_reference_fixtures(api, golden, fixture_dir, db, form, tmp_path):
    rels = golden[1]["K8_inputs"]["dbs"][db]
    texts = [read(os.path.join(fixture_dir, r)) for r in rels]
    paths = write_texts(tmp_path, db, texts, form)
    sets = [api.RegionSet(p) for p in paths]
    names = [os.path.basename(r) for r in rels]
    p = same_as_host_writer(api, build(api, paths, form), sets, names, tmp_path, db)
    # default names: set{i} over the database's files
    build(api, paths, form).save(str(tmp_path / "default.igd"))
    api.write_igd_file(sets, [f"set{i}" for i in range(len(sets))], str(tmp_path / "default_host.igd"))
    assert read(str(tmp_path / "default.tsv")) == read(str(tmp_path / "default_host.tsv"))
    # round trip: a database loaded from the file writes the same file again
    api.Igd.from_igd_file(p).save(str(tmp_path / "again.igd"), names)
    assert read(str(tmp_path / "again.igd")) == read(p)


LONG = "chrLong_" + "x" * 45  # cut to 40 bytes in the file
EDGE = [
    # text order of the names differs from their sorted order; chrZ spans five tiles; tile-boundary starts and ends
    f"chrZ\t0\t70000\nchrB\t16384\t32768\nchrB\t16384\t32769\nchrB\t100\t200\nchrB\t100\t300\nchrA\t5\t5\n"
    f"chrA\t10\t3000000000\nchrDropped\t2147483648\t2147483700\n{LONG}\t1\t2\nchrB\t32767\t32768\nchrZ\t65536\t65537\n",
    "chrB\t50\t40\nchrB\t7\t7\n",  # every line dropped: 0 regions, 0.00
    f"chrB\t100\t150\nchrC\t0\t16385\nchrA\t16383\t16384\nchrZ\t3\t131072\nchrDropped\t9\t9\nchrA\t16383\t16390\n{LONG}\t0\t1\n",
    "chrC\t4294967290\t4294967295\nchrC\t0\t1\n",
]


@pytest.mark.parametrize("form", FORMS)
def test_edge_database(api, form, tmp_path):
    paths = write_texts(tmp_path, "edge", [t.encode() for t in EDGE], form)
    sets = [api.RegionSet(p) for p in paths]
    names = [f"edge{i}" for i in range(len(paths))]
    p = same_as_host_writer(api, build(api, paths, form), sets, names, tmp_path, "edge")
    b = read(p)
    n_ctg = int.from_bytes(b[8:12], "little")
    tiles = [int.from_bytes(b[12 + 4 * i:16 + 4 * i], "little") for i in range(n_ctg)]
    nb = 12 + 4 * n_ctg + 4 * sum(tiles)
    ctg = [b[nb + 40 * i:nb + 40 * (i + 1)].rstrip(b"\0").decode() for i in range(n_ctg)]
    # file 0 keeps chrB, chrLong.., chrZ (chrA only has dropped lines there); file 2 adds chrA and chrC
    assert ctg == ["chrB", LONG[:40], "chrZ", "chrA", "chrC"]
    assert tiles == [3, 1, 8, 2, 2]
    tsv = read(p[:-4] + ".tsv").decode().splitlines()
    assert tsv[2] == "1\tedge1\t0\t0.00"
    api.Igd.from_igd_file(p).save(str(tmp_path / "again.igd"), names)
    assert read(str(tmp_path / "again.igd")) == b


def test_unsorted_region_lists(api, tmp_path):
    """RegionSets made from lists keep their order: contigs follow insertion, as the host writer's"""
    rng = np.random.default_rng(5)
    chroms = ["chr9", "chr1", "chrX", "chr10", "chr2"]
    sets = []
    for f in range(5):
        regs = []
        for _ in range(400):
            s = int(rng.integers(0, 200_000))
            regs.append((chroms[int(rng.integers(0, len(chroms)))], s, s + int(rng.integers(0, 40_000))))
        sets.append(api.RegionSet(regs))
    names = [f"u{i}" for i in range(len(sets))]
    same_as_host_writer(api, api.Igd(sets), sets, names, tmp_path, "unsorted")


def sorted_per_file(c, s, e, n_files, per):
    """records stably sorted per file by (name bytes, start), as RegionSet::try_from orders a file"""
    from gtars_b200 import synth
    rank = np.argsort(np.argsort(np.array([n.encode() for n in synth.CHROM_NAMES[:25]], dtype=object)))
    f = np.repeat(np.arange(n_files), per)
    o = np.lexsort((s, rank[c], f))
    return c[o], s[o], e[o]


def test_scale_through_ffi(ctx, tmp_path):
    """2 000 BED files x 2e4 regions: the device's bytes == the oracle's bulk writer; the .tsv numbers == numpy"""
    from gtars_b200 import ffi, synth
    from oracle import oracle as orc
    n_files, per = 2000, 20000
    c, s, e = synth_db(n_files, per, 21)
    text = bed_text(c, s, e)
    line_end = np.flatnonzero(text == 10) + 1
    fo = np.concatenate([[0], line_end[per - 1::per]]).astype(np.uint64)
    g, names = ffi.Igd.from_bed_text(ctx, text, fo)
    del text
    got, regions, widths = g.save_bytes(names)
    g.close()
    kept = s < e
    assert np.array_equal(regions, kept.reshape(n_files, per).sum(1))
    assert np.array_equal(widths, np.where(kept, e.astype(np.int64) - s, 0).reshape(n_files, per).sum(1).astype(np.uint64))
    sc, ss, se = sorted_per_file(c, s, e, n_files, per)
    p = str(tmp_path / "scale.igd")
    orc.Igd(np.arange(0, n_files * per + 1, per, dtype=np.uint64), sc, ss, se).save(p, synth.CHROM_NAMES[:25])
    assert got.tobytes() == read(p)


def test_payload_past_2_gib(ctx, tmp_path):
    """1e7 records of ~15 tiles each: more than 2^31 bytes of records, equal to the oracle writer by SHA-256"""
    from gtars_b200 import ffi, synth
    from oracle import oracle as orc
    n_files, per = 10, 1_000_000
    rng = np.random.default_rng(8)
    n = n_files * per
    c = rng.integers(0, 25, n).astype(np.uint32)
    s = rng.integers(0, 2**30, n).astype(np.uint32)
    e = (s + rng.integers(14 * NBP, 16 * NBP, n)).astype(np.uint32)
    fo = np.arange(0, n + 1, per, dtype=np.uint64)
    g = ffi.Igd(ctx, fo, 25, c, s, e)
    got, regions, _ = g.save_bytes(synth.CHROM_NAMES[:25])
    g.close()
    entries = int(((e - 1) // NBP - s // NBP + 1).astype(np.int64).sum())
    assert entries * 16 > 2**31 and np.array_equal(regions, np.full(n_files, per))
    want_sha = hashlib.sha256(got).hexdigest()
    del got
    p = str(tmp_path / "big.igd")
    orc.Igd(fo, c, s, e).save(p, synth.CHROM_NAMES[:25])
    h = hashlib.sha256()
    with open(p, "rb") as f:
        for block in iter(lambda: f.read(1 << 26), b""):
            h.update(block)
    os.remove(p)
    assert h.hexdigest() == want_sha


def test_multi_device_context_equals_single(ctx):
    from gtars_b200 import ffi
    if ffi.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    n_files, per = 37, 3000
    c, s, e = synth_db(n_files, per, 11)
    e[5::997] = s[5::997] + 5 * NBP
    texts = [bed_text(c[f * per:(f + 1) * per], s[f * per:(f + 1) * per], e[f * per:(f + 1) * per]).tobytes() for f in range(n_files)]
    fo = np.cumsum([0] + [len(t) for t in texts]).astype(np.uint64)
    ro = np.arange(0, n_files * per + 1, per, dtype=np.uint64)
    multi = ffi.Context(devices=[0, 1])
    one, names = ffi.Igd.from_bed_text(ctx, b"".join(texts), fo)
    two, names2 = ffi.Igd.from_bed_text(multi, b"".join(texts), fo)
    assert names2 == names
    for a, b in zip(one.save_bytes(names), two.save_bytes(names)):
        assert np.array_equal(a, b)
    one_a, two_a = ffi.Igd(ctx, ro, 25, c, s, e), ffi.Igd(multi, ro, 25, c, s, e)
    from gtars_b200 import synth
    for a, b in zip(one_a.save_bytes(synth.CHROM_NAMES[:25]), two_a.save_bytes(synth.CHROM_NAMES[:25])):
        assert np.array_equal(a, b)
    for g in (one, two, one_a, two_a):
        g.close()
    multi.close()


def test_errors_leave_the_context_usable(api, ctx, tmp_path):
    from gtars_b200 import ffi
    sets = [api.RegionSet([("chr1", 0, 100), ("chr2", 5, 50000)])]
    with pytest.raises(api.GtarsError, match="database"):
        api.Igd.from_single_region_set(sets[0]).save(str(tmp_path / "single.igd"))
    g = ffi.Igd(ctx, [0, 2], 2, [0, 1], [0, 5], [100, 50000])
    with pytest.raises(ffi.GtarsGpuError) as ei:
        g.save_bytes(["chr1"])
    assert ei.value.code == 1
    bad = str(tmp_path / "no_such_dir" / "db.igd")
    with pytest.raises(api.GtarsError, match="no_such_dir"):
        api.Igd(sets).save(bad)
    got, regions, widths = g.save_bytes(["chr1", "chr2"])
    g.close()
    api.write_igd_file(sets, ["set0"], str(tmp_path / "host.igd"))
    assert got.tobytes() == read(str(tmp_path / "host.igd"))
    assert regions.tolist() == [2] and widths.tolist() == [100 + 49995]
