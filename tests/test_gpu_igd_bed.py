"""An IGD database from its BED files parsed on the device (gtgpu_igd_build_bed / _gz, ffi.Igd.from_bed_text / from_bed_gz,
api.Igd.from_bed_files) answers every count exactly as Igd([RegionSet(p) for p in paths]) built from the host parser does:
plain text, one gzip member per file, BGZF, and a mix of plain and .gz paths, in windows of GTGPU_INGEST_WINDOW bytes."""
import gzip
import os
import re

import numpy as np
import pytest

from tests.test_gpu_fragment_file_text import bgzf_fast
from tests.test_gpu_score_text import bgzf

pytestmark = pytest.mark.gpu

FORMS = ("plain", "gzip", "bgzf", "mixed")


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


def write_files(d, name, texts, form):
    """texts as files of one form; "mixed" alternates plain and single-member gzip paths."""
    paths = []
    for i, t in enumerate(texts):
        kind = form if form != "mixed" else ("plain", "gzip")[i % 2]
        p = str(d / (f"{name}_{form}_{i:05d}.bed" + ("" if kind == "plain" else ".gz")))
        with open(p, "wb") as f:
            f.write(t if kind == "plain" else gzip.compress(t, mtime=0) if kind == "gzip" else bgzf(t))
        paths.append(p)
    return paths


def queries_over(names, rng, per_name=6):
    """query sets over every chromosome named (and one unknown name): wide, narrow and touching regions"""
    sets = []
    for n in list(names) + ["chrNowhere"]:
        q = [(n, 0, 2**31 - 1), (n, 0, 1)]
        for _ in range(per_name):
            s = int(rng.integers(0, 3000))
            q.append((n, s, s + int(rng.integers(1, 400))))
        sets.append(q)
    sets.append([r for q in sets for r in q])
    return sets


def matrices(igd, sets, m=1):
    return igd._count(sets, m, True), igd._count(sets, m, False)


def same_as_host(api, paths, names, seed=0, also=()):
    """api.Igd.from_bed_files(paths) == api.Igd([RegionSet(p) ...]) on queries over every name; returns the device matrices"""
    dev = api.Igd.from_bed_files(paths)
    host = api.Igd([api.RegionSet(p) for p in paths])
    sets = queries_over(names, np.random.default_rng(seed)) + list(also)
    for m in (1, 7):
        for a, b in zip(matrices(dev, sets, m), matrices(host, sets, m)):
            assert np.array_equal(a, b), (paths[:2], m)
    di, hi = dev.info(), host.info()
    assert (di["n_files"], di["n_records"]) == (hi["n_files"], hi["n_records"]) == (len(paths), di["n_records"])
    return matrices(dev, sets)


def text_form(ctx, texts):
    """ffi.Igd.from_bed_text over the texts back to back, and from_bed_gz over one gzip member per file: same names"""
    from gtars_b200 import ffi
    fo = np.cumsum([0] + [len(t) for t in texts]).astype(np.uint64)
    g, names = ffi.Igd.from_bed_text(ctx, b"".join(texts), fo)
    members = [gzip.compress(t, mtime=0) for t in texts]
    mo = np.cumsum([0] + [len(m) for m in members]).astype(np.uint64)
    gg, names_gz = ffi.Igd.from_bed_gz(ctx, b"".join(members), np.arange(len(texts) + 1), mo)
    assert names_gz == names and gg.info()["n_records"] == g.info()["n_records"]
    gg.close()
    return g, names


def first_appearance(texts):
    """chromosome names in first-appearance order over the region lines (header rule per file)"""
    seen = []
    for t in texts:
        for i, line in enumerate(t.decode().split("\n")):
            line = line.rstrip("\r")
            if line.startswith(("browser", "track", "#")):
                continue
            f = line.split("\t")
            if len(f) < 3 or not f[1].lstrip("+").isdigit():
                continue  # a header (first line) here; the edge texts have no other non-region line
            if f[0] not in seen:
                seen.append(f[0])
    return seen


def edge_texts():
    rng = np.random.default_rng(5)

    def lines(names, n):
        out = []
        for _ in range(n):
            s = int(rng.integers(0, 3000))
            out.append(f"{names[int(rng.integers(0, len(names)))]}\t{s}\t{s + int(rng.integers(1, 500))}")
        return out

    base = ["chr1", "chr2", "chrX"]
    c = {}
    c["header_in_file_3"] = [("\n".join(lines(base, 30)) + "\n").encode() for _ in range(3)] + [
        ("chrom\tstart\tend\n" + "\n".join(lines(base, 30)) + "\n").encode(),
        ("chrom\tchromStart\tchromEnd\tname\n" + "\n".join(lines(base, 5)) + "\n").encode()]
    c["comments_crlf"] = [("browser position chr1:1-100\r\ntrack name=x\r\n# c\r\n" + "\r\n".join(lines(base, 40)) + "\r\n").encode(),
                          ("#only a comment first\n" + "\n".join(lines(base, 40)) + "\n#end\n").encode(),
                          ("\r\n".join(lines(base, 10)) + "\r\n").encode()]
    c["no_final_newline"] = [("\n".join(lines(base, 20))).encode(), ("\n".join(lines(base, 20))).encode(),
                             ("\n".join(lines(base, 20)) + "\n").encode(), b"chr2\t5\t10"]
    c["dropped_records"] = [("chr1\t100\t100\nchr1\t300\t200\nchr1\t2147483648\t2147483700\nchr2\t4294967290\t4294967295\n"
                             "chrDropOnly\t50\t10\n" + "\n".join(lines(base, 20)) + "\n").encode(),
                            ("\n".join(lines(base, 20)) + "\n").encode()]
    c["late_and_prefix_names"] = [("\n".join(lines(base, 20)) + "\n").encode(),
                                  ("\n".join(lines(["chr1", "chr10", "chr1_random", "chr100"], 40)) + "\n").encode(),
                                  ("\n".join(lines(["chrLate"], 5) + lines(base, 5)) + "\n").encode()]
    c["one_file"] = [("\n".join(lines(base + ["chrM"], 200)) + "\n").encode()]
    c["tiny_files"] = [("\n".join(lines(base + [f"scaf{i % 97}"], 1 + i % 3)) + ("\n" if i % 4 else "")).encode() for i in range(5000)]
    return c


@pytest.mark.parametrize("form", FORMS)
def test_reference_fixtures(api, golden, fixture_dir, form, tmp_path):
    """igd_file_list_01 / _02 and lola_multi_db: the K7 known answer, query1 / query2 / all-vs-all and lola_contingency equal
    the host-built database."""
    k8 = golden[1]["K8_inputs"]
    for case in golden[1]["K7_igd_sets"]:
        if "db_files" in case:
            texts = [open(os.path.join(fixture_dir, f), "rb").read() for f in case["db_files"]]
            db = api.Igd.from_bed_files(write_files(tmp_path, "k7", texts, form))
            assert db.count_set_overlaps([tuple(r) for r in case["query"]], case["min_overlap"]) == case["set_overlaps"], case["cite"]
    for name, rels in k8["dbs"].items():
        texts = [open(os.path.join(fixture_dir, r), "rb").read() for r in rels]
        paths = write_files(tmp_path, name, texts, form)
        sets = [api.RegionSet(p) for p in paths]
        queries = [api.RegionSet(os.path.join(fixture_dir, q)) for q in k8["queries"]] + sets
        dev = api.Igd.from_bed_files(paths)
        host = api.Igd(sets)
        for m in (1, 10):
            for a, b in zip(matrices(dev, queries, m), matrices(host, queries, m)):
                assert np.array_equal(a, b), (name, m)
        assert [dev.info()[k] for k in ("n_files", "n_records")] == [host.info()[k] for k in ("n_files", "n_records")]
        universe = api.RegionSet(os.path.join(fixture_dir, k8["queries"][0]))
        assert np.array_equal(api.lola_contingency(dev, queries[1:], universe), api.lola_contingency(host, queries[1:], universe))


@pytest.mark.parametrize("form", FORMS)
@pytest.mark.parametrize("case", sorted(edge_texts()))
def test_edge_files(api, ctx, case, form, tmp_path):
    texts = edge_texts()[case]
    if case == "tiny_files" and form in ("gzip", "mixed"):
        texts = texts[:1000]  # single-member gzip of every file is the host's zlib speed, not the device's
    names = first_appearance(texts)
    paths = write_files(tmp_path, case, texts, form)
    same_as_host(api, paths, names)
    if form == "plain":
        g, got = text_form(ctx, texts)
        assert got == names                         # ids in first-appearance order, dropped-only names included
        assert g.info()["n_files"] == len(texts)
        g.close()


def test_forced_windows(api, ctx, tmp_path, monkeypatch):
    """Windows of 1 byte to 64 KiB give the default window's matrices, including file boundaries exactly on window cuts (every
    file of "aligned" is 64 bytes) and files whose last line has no '\\n'."""
    from gtars_b200 import ffi
    texts = edge_texts()
    rng = np.random.default_rng(8)
    aligned = []
    for i in range(40):
        s = int(rng.integers(0, 3000))
        line = f"chr{1 + i % 3}\t{s:010d}\t{s + 50:010d}"            # 4 + 1 + 10 + 1 + 10 = 26 bytes
        aligned.append((line + "\n" + line[:-1] + "7" + "\t" + "x" * 9 + "\n").encode())
    assert all(len(t) == 64 for t in aligned)
    dbs = {"aligned": aligned, "no_final_newline": texts["no_final_newline"], "comments_crlf": texts["comments_crlf"],
           "header_in_file_3": texts["header_in_file_3"], "tiny": texts["tiny_files"][:300]}
    paths = {k: write_files(tmp_path, k, v, "bgzf") + write_files(tmp_path, k, v, "plain") for k, v in dbs.items()}
    monkeypatch.delenv("GTGPU_INGEST_WINDOW", raising=False)
    want = {k: same_as_host(api, paths[k][len(dbs[k]):], first_appearance(dbs[k])) for k in dbs}
    for w in ("1", "7", "64", "1024", "65536"):
        monkeypatch.setenv("GTGPU_INGEST_WINDOW", w)
        for k, v in dbs.items():
            for half in (paths[k][:len(v)], paths[k][len(v):]):
                got = matrices(api.Igd.from_bed_files(half), queries_over(first_appearance(v), np.random.default_rng(0)))
                assert all(np.array_equal(a, b) for a, b in zip(got, want[k])), (w, k, half[0])
            fo = np.cumsum([0] + [len(t) for t in v]).astype(np.uint64)
            g, names = ffi.Igd.from_bed_text(ctx, b"".join(v), fo)
            assert names == first_appearance(v), (w, k)
            g.close()


def _file_line(msg):
    m = re.search(r"file (\d+), line (\d+)", msg)
    assert m, msg
    return int(m.group(1)), int(m.group(2))


def test_errors_name_file_and_line(api, ctx, tmp_path, monkeypatch):
    from gtars_b200 import ffi
    rng = np.random.default_rng(9)
    good = [("\n".join(f"chr{1 + j % 2}\t{int(rng.integers(0, 5000))}\t6000" for j in range(300)) + "\n").encode() for _ in range(6)]
    fo = np.cumsum([0] + [len(t) for t in good]).astype(np.uint64)
    ref, ref_names = ffi.Igd.from_bed_text(ctx, b"".join(good), fo)
    q = (np.array([0, 2], dtype=np.uint64), [0, 1], [0, 0], [10000, 10000])
    want = ref.count_set_overlaps(*q)

    def still_usable():
        g, names = ffi.Igd.from_bed_text(ctx, b"".join(good), fo)
        assert names == ref_names and np.array_equal(g.count_set_overlaps(*q), want)
        g.close()

    # (a malformed first line of a file is that file's header row, so the earliest error is on line 2)
    for k, j, window in ((0, 2, None), (3, 17, None), (5, 290, "4096"), (4, 300, "1")):
        if window:
            monkeypatch.setenv("GTGPU_INGEST_WINDOW", window)
        lines = good[k].decode().split("\n")
        lines[j - 1] = "chr1\tabc\t100"
        bad = list(good)
        bad[k] = "\n".join(lines).encode()
        bfo = np.cumsum([0] + [len(t) for t in bad]).astype(np.uint64)
        members = [gzip.compress(t, mtime=0) for t in bad]
        mo = np.cumsum([0] + [len(m) for m in members]).astype(np.uint64)
        for call in (lambda: ffi.Igd.from_bed_text(ctx, b"".join(bad), bfo),
                     lambda: ffi.Igd.from_bed_gz(ctx, b"".join(members), np.arange(len(bad) + 1), mo)):
            with pytest.raises(ffi.GtarsGpuError) as e:
                call()
            assert e.value.code == 1 and _file_line(str(e.value)) == (k, j), str(e.value)
            still_usable()
        paths = write_files(tmp_path, f"bad{k}", bad, "mixed")
        with pytest.raises(api.GtarsError) as e:
            api.Igd.from_bed_files(paths)
        assert paths[k] in str(e.value) and f"line {j}" in str(e.value), str(e.value)
        monkeypatch.delenv("GTGPU_INGEST_WINDOW", raising=False)
    for empty in (b"", b"# only\n#comments\ntrack x\n", b"chrom\tstart\tend\n"):
        texts = good[:2] + [empty] + good[2:]
        efo = np.cumsum([0] + [len(t) for t in texts]).astype(np.uint64)
        with pytest.raises(ffi.GtarsGpuError) as e:
            ffi.Igd.from_bed_text(ctx, b"".join(texts), efo)
        assert e.value.code == 1 and "file 2: " in str(e.value) and "0 regions" in str(e.value)
        still_usable()
        for form in ("plain", "gzip"):
            paths = write_files(tmp_path, "empty", texts, form)
            with pytest.raises(api.GtarsError) as e:
                api.Igd.from_bed_files(paths)
            assert paths[2] in str(e.value) and "0 regions" in str(e.value)
    ref.close()


def test_final_cr_follows_the_device_parser(ctx):
    """A last line ending in '\\r' without '\\n' is malformed, as gtgpu_parse_bed has it (the host reader strips the '\\r')."""
    from gtars_b200 import ffi
    t = b"chr1\t1\t10\nchr1\t5\t20\r"
    n = ffi.C.c_uint64(0)
    h = [ffi.C.c_void_p() for _ in range(3)]
    blob, offs = ffi._names_blob(["chr1"])
    st = ffi.lib().gtgpu_parse_bed(ctx._h, t, len(t), 1, blob, ffi._p(offs), ffi.C.byref(n), *(ffi.C.byref(x) for x in h))
    assert st == 1
    for texts in ([t], [b"chr2\t1\t5\n", t], [t, b"chr2\t1\t5\n"]):
        fo = np.cumsum([0] + [len(x) for x in texts]).astype(np.uint64)
        with pytest.raises(ffi.GtarsGpuError) as e:
            ffi.Igd.from_bed_text(ctx, b"".join(texts), fo)
        assert _file_line(str(e.value)) == (texts.index(t), 2)


def bed_text(chr_id, start, end):
    """Vectorised BED lines "name\\tSTART\\tEND\\n" (10-digit zero-padded coordinates) as a uint8 array."""
    from gtars_b200 import synth
    names = [n.encode() for n in synth.CHROM_NAMES]
    tab = np.zeros((len(names), 8), dtype=np.uint8)
    for i, n in enumerate(names):
        tab[i, :len(n)] = list(n)
    nl = np.array([len(n) for n in names], dtype=np.int64)[chr_id]
    off = np.zeros(len(chr_id) + 1, dtype=np.int64)
    np.cumsum(nl + 23, out=off[1:])
    out = np.empty(int(off[-1]), dtype=np.uint8)
    a = off[:-1]
    for j in range(int(nl.max())):
        m = nl > j
        out[a[m] + j] = tab[chr_id[m], j]
    p = a + nl
    out[p], out[p + 11], out[p + 22] = 9, 9, 10
    for col, v in ((p + 1, start), (p + 12, end)):
        v = np.asarray(v).astype(np.uint64)
        for j in range(9, -1, -1):
            out[col + j] = (v % 10).astype(np.uint8) + 48
            v //= 10
    return out


def synth_db(n_files, per_file, seed):
    rng = np.random.default_rng(seed)
    n = n_files * per_file
    c = rng.integers(0, 25, n).astype(np.int64)
    s = rng.integers(0, 2**28, n).astype(np.uint32)
    e = (s + rng.integers(1, 5000, n)).astype(np.uint32)
    e[::1000] = s[::1000]                                               # a few records the IGD drops
    return c, s, e


def query_batch(seed, n_sets=64, per_set=2000):
    rng = np.random.default_rng(seed)
    n = n_sets * per_set
    c = rng.integers(0, 26, n).astype(np.uint32)                        # id 25 names no chromosome
    s = rng.integers(0, 2**28, n).astype(np.uint32)
    return np.arange(0, n + 1, per_set, dtype=np.uint64), c, s, (s + rng.integers(1, 20000, n)).astype(np.uint32)


def same_counts(a, names, b, q):
    """a (chromosome ids through `names`) and b (ids = synth.CHROM_NAMES positions) give equal matrices for the batch q"""
    from gtars_b200 import synth
    idx = {n: i for i, n in enumerate(names)}
    remap = np.array([idx.get(n, 0xFFFFFFFF) for n in synth.CHROM_NAMES[:25]] + [0xFFFFFFFF], dtype=np.uint32)
    so, c, s, e = q
    assert np.array_equal(a.count_set_overlaps(so, remap[c], s, e), b.count_set_overlaps(so, c, s, e))
    assert np.array_equal(a.count_region_hits(so, remap[c], s, e), b.count_region_hits(so, c, s, e))


def test_c4_shape_reduced(ctx):
    """2 000 sets x 2e4 regions (C4's shape at a fifth of its sets) as BED text == ffi.Igd from the same arrays; and as BGZF."""
    from gtars_b200 import ffi
    n_files, per = 2000, 20000
    c, s, e = synth_db(n_files, per, 3)
    text = bed_text(c, s, e)
    line_end = np.flatnonzero(text == 10) + 1
    fo = np.concatenate([[0], line_end[per - 1::per]]).astype(np.uint64)
    g, names = ffi.Igd.from_bed_text(ctx, text, fo)
    ref = ffi.Igd(ctx, np.arange(0, n_files * per + 1, per, dtype=np.uint64), 25, c, s, e)
    assert g.info()["n_records"] == ref.info()["n_records"]
    q = query_batch(4)
    same_counts(g, names, ref, q)
    g.close()
    gz, mo, fm = [], [np.zeros(1, dtype=np.uint64)], [0]                 # BGZF per file, the files back to back
    base = 0
    for f in range(n_files):
        b = bgzf_fast(text[int(fo[f]):int(fo[f + 1])].tobytes())
        gz.append(b)
        mo.append(ffi.gzip_members(b)[1:] + np.uint64(base))
        fm.append(fm[-1] + len(mo[-1]))
        base += len(b)
    g, names = ffi.Igd.from_bed_gz(ctx, b"".join(gz), np.array(fm, dtype=np.uint64), np.concatenate(mo))
    same_counts(g, names, ref, q)
    g.close()
    ref.close()


def test_text_past_4_gib(ctx):
    """A text of more than 4.4 GB (18 files of 1e7 regions) through the ffi, in the default 2 GiB windows."""
    from gtars_b200 import ffi
    per, reps = 10_000_000, 18
    c, s, e = synth_db(1, per, 6)
    chunk = bed_text(c, s, e)
    text = np.tile(chunk, reps)
    assert text.nbytes > 4.4e9
    fo = np.arange(reps + 1, dtype=np.uint64) * np.uint64(chunk.nbytes)
    g, names = ffi.Igd.from_bed_text(ctx, text, fo)
    del text
    ref = ffi.Igd(ctx, np.arange(reps + 1, dtype=np.uint64) * np.uint64(per), 25, np.tile(c, reps), np.tile(s, reps), np.tile(e, reps))
    assert g.info()["n_records"] == ref.info()["n_records"]
    same_counts(g, names, ref, query_batch(7, 16, 4000))
    g.close()
    ref.close()


def test_multi_device_context_equals_single(ctx):
    from gtars_b200 import ffi
    if ffi.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    n_files, per = 37, 3000
    c, s, e = synth_db(n_files, per, 11)
    texts = [bed_text(c[f * per:(f + 1) * per], s[f * per:(f + 1) * per], e[f * per:(f + 1) * per]).tobytes() for f in range(n_files)]
    fo = np.cumsum([0] + [len(t) for t in texts]).astype(np.uint64)
    one, names = ffi.Igd.from_bed_text(ctx, b"".join(texts), fo)
    multi = ffi.Context(devices=[0, 1])
    two, names2 = ffi.Igd.from_bed_text(multi, b"".join(texts), fo)
    assert names2 == names and two.info()["n_records"] == one.info()["n_records"]
    so, qc, qs, qe = query_batch(12, 8, 1000)
    qc = np.minimum(qc, len(names) - 1).astype(np.uint32)
    for fn in ("count_set_overlaps", "count_region_hits"):
        assert np.array_equal(getattr(two, fn)(so, qc, qs, qe), getattr(one, fn)(so, qc, qs, qe))
    two.close()
    one.close()
    multi.close()


def gz_members(texts):
    """one gzip member per text: (bytes, file_members, member_offsets) for ffi.Igd.from_bed_gz"""
    members = [gzip.compress(t, mtime=0) for t in texts]
    return b"".join(members), np.arange(len(texts) + 1), np.cumsum([0] + [len(m) for m in members]).astype(np.uint64)


def test_names_first_seen_over_many_windows(ctx, monkeypatch):
    """1e5 distinct chromosome names, first seen all along the text, in windows of 64 KiB (about 100 windows): the name table
    grows during the call.  Names and counts equal gtgpu_igd_build on the same records with first-appearance ids."""
    from gtars_b200 import ffi
    n_names, n_files, per = 100_000, 30, 10_000
    n = n_files * per
    rng = np.random.default_rng(21)
    c = np.arange(n) * n_names // n                                     # every name, first seen in order along the text
    c[1::3] = (c[1::3] + rng.integers(0, 4, len(c[1::3]))) % n_names  # and some lines a few names ahead
    s = rng.integers(0, 100_000, n).astype(np.uint32)
    e = (s + rng.integers(1, 5000, n)).astype(np.uint32)
    lines = [f"c{a}\t{b}\t{d}\n" for a, b, d in zip(c.tolist(), s.tolist(), e.tolist())]
    texts = ["".join(lines[f * per:(f + 1) * per]).encode() for f in range(n_files)]
    u, first = np.unique(c, return_index=True)
    assert len(u) == n_names
    order = u[np.argsort(first)]                                        # name of id i, in first-appearance order
    id_of = np.empty(n_names, dtype=np.uint32)
    id_of[order] = np.arange(n_names, dtype=np.uint32)
    ref = ffi.Igd(ctx, np.arange(0, n + 1, per, dtype=np.uint64), n_names, id_of[c], s, e)
    so = np.arange(0, 64 * 500 + 1, 500, dtype=np.uint64)
    qc = rng.integers(0, n_names, 64 * 500).astype(np.uint32)
    qs = rng.integers(0, 100_000, 64 * 500).astype(np.uint32)
    qe = (qs + rng.integers(1, 20_000, 64 * 500)).astype(np.uint32)
    fo = np.cumsum([0] + [len(t) for t in texts]).astype(np.uint64)
    monkeypatch.setenv("GTGPU_INGEST_WINDOW", "65536")
    for g, names in (ffi.Igd.from_bed_text(ctx, b"".join(texts), fo), ffi.Igd.from_bed_gz(ctx, *gz_members(texts))):
        assert names == [f"c{v}" for v in order]
        assert g.info()["n_records"] == ref.info()["n_records"]
        for fn in ("count_set_overlaps", "count_region_hits"):
            assert np.array_equal(getattr(g, fn)(so, qc, qs, qe), getattr(ref, fn)(so, qc, qs, qe)), fn
        g.close()
    ref.close()


def test_name_limit(ctx):
    """262 144 distinct chromosome names load; one more is GTGPU_ERR_UNSUPPORTED with its message, and the ctx stays usable."""
    from gtars_b200 import ffi
    limit = 262_144
    for n_names in (limit, limit + 1):
        lines = [f"n{i}\t{i % 1000}\t{i % 1000 + 10}\n" for i in range(n_names)]
        texts = ["".join(lines[f::4]).encode() for f in range(4)]
        fo = np.cumsum([0] + [len(t) for t in texts]).astype(np.uint64)
        for call in (lambda: ffi.Igd.from_bed_text(ctx, b"".join(texts), fo), lambda: ffi.Igd.from_bed_gz(ctx, *gz_members(texts))):
            if n_names == limit:
                g, names = call()
                assert len(names) == limit and names[:3] == ["n0", "n4", "n8"] and g.info()["n_records"] == limit
                g.close()
            else:
                with pytest.raises(ffi.GtarsGpuError) as err:
                    call()
                assert err.value.code == 6 and "more than 262144 distinct chromosome names" in str(err.value), str(err.value)
    g, names = ffi.Igd.from_bed_text(ctx, b"chr1\t1\t5\n", np.array([0, 9], dtype=np.uint64))
    assert names == ["chr1"]
    g.close()
