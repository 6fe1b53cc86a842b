"""A batch of BED files tokenized in one device pass (gtgpu_tokenize_bed_files / _gz, ffi.Index.tokenize_bed_files,
api.Tokenizer.encode_bed_files) gives, file by file, what encode_bed_file(path) and encode(RegionSet(path)) give: reference
vectors, edge files in every form (plain, one gzip member per file, BGZF, plain and gzip mixed), forced windows, errors that
name the file and line, C2-shaped batches sorted and shuffled, a text past 4 GiB, and a multi-device ctx."""
import gzip
import json
import os
import re
import subprocess
import sys

import numpy as np
import pytest

from tests.test_gpu_igd_bed import FORMS, bed_text, edge_texts, write_files

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
gpu = pytest.mark.gpu
NAMES = ["chr1", "chr2", "chrX", "chr10", "chr1_random", "chr100", "chrM", "chrLate"] + [f"scaf{i}" for i in range(0, 97, 3)]


@pytest.fixture(scope="module")
def api():
    from gtars_b200 import api as a
    a.device(0)
    return a


@pytest.fixture(scope="module")
def toks(api, tmp_path_factory):
    """Bits (from the BED file) and AIList (from a config) tokenizers over one universe of overlapping peaks on NAMES."""
    d = tmp_path_factory.mktemp("universe")
    rng = np.random.default_rng(17)
    lines = []
    for _ in range(3000):
        s = int(rng.integers(0, 3400))
        lines.append(f"{NAMES[int(rng.integers(0, len(NAMES)))]}\t{s}\t{s + int(rng.integers(20, 400))}")
    (d / "universe.bed").write_text("\n".join(lines) + "\n")
    (d / "ailist.toml").write_text('universe = "universe.bed"\ntokenizer_type = "ailist"\n')
    return api.Tokenizer(str(d / "universe.bed")), api.Tokenizer.from_config(str(d / "ailist.toml"))


def local_texts():
    """files out of order next to sorted ones, and equal (name, start) pairs whose order only stability decides"""
    rng = np.random.default_rng(23)
    names = ["chr1", "chr10", "chr2", "chrX", "chr1_random", "chrNowhere"]
    mixed = []
    for i in range(12):
        rows = [(names[int(rng.integers(0, len(names)))], int(rng.integers(0, 3000))) for _ in range(60)]
        if i % 2:
            rows.sort()
        mixed.append("".join(f"{c}\t{s}\t{s + 1 + (7 * k) % 300}\n" for k, (c, s) in enumerate(rows)).encode())
    ties = []
    for i in range(6):
        rows = [(names[int(rng.integers(0, 3))], 100 * int(rng.integers(0, 20))) for _ in range(80)]
        ties.append("".join(f"{c}\t{s}\t{s + 1 + int(rng.integers(0, 600))}\n" for c, s in rows).encode())
    return {"sorted_and_unsorted": mixed, "equal_starts": ties}


def all_cases():
    return {**edge_texts(), **local_texts()}


def same_as_existing_paths(api, toks, paths, per_file=True):
    """encode_bed_files(paths)[f] == encode_bed_file(paths[f]) == encode(RegionSet(paths[f])), Bits and AIList"""
    for tok in toks:
        got = tok.encode_bed_files(paths)
        assert len(got) == len(paths)
        assert got == tok.encode_batch([api.RegionSet(p) for p in paths]), paths[0]
        if per_file or tok is toks[0]:                                 # (AIList per file: not over thousands of files)
            assert got == [tok.encode_bed_file(p) for p in paths], paths[0]
    return toks[0].encode_bed_files(paths)


@gpu
def test_reference_vectors(api, fixture_dir, tmp_path):
    """K5 / D1: to_tokenize.bed against peaks.bed is [22, 23, 24] with Bits, [22, 24, 23] with AIList; a file without a hit is
    [unk]; all in one batch, with the same files repeated, plain and .gz."""
    uni = os.path.join(fixture_dir, "tokenizers", "peaks.bed")
    q = os.path.join(fixture_dir, "to_tokenize.bed")
    qgz = str(tmp_path / "to_tokenize.bed.gz")
    open(qgz, "wb").write(gzip.compress(open(q, "rb").read(), mtime=0))
    miss = str(tmp_path / "miss.bed")
    open(miss, "w").write("chrNope\t1\t2\nchr1\t1\t2\n")
    toml = os.path.join(fixture_dir, "tokenizers", "tokenizer_ailist_batch.toml")
    open(toml, "w").write('universe = "peaks.bed.gz"\ntokenizer_type = "ailist"\n')
    for tok, want in ((api.Tokenizer(uni), [22, 23, 24]), (api.Tokenizer.from_config(toml), [22, 24, 23])):
        unk = [tok.unk_token_id]
        assert tok.encode_bed_files([q]) == [want]
        assert tok.encode_bed_files([qgz]) == [want]                     # every path .gz: inflated on the device
        assert tok.encode_bed_files([miss]) == [unk]
        batch = [q, miss, uni, qgz, q, miss, q]
        assert tok.encode_bed_files(batch) == [want, unk, tok.encode_bed_file(uni), want, want, unk, want]
        assert tok.encode_bed_files([qgz, uni + ".gz", qgz]) == [want, tok.encode(api.RegionSet(uni)), want]
        assert tok.encode_bed_files([]) == []


@gpu
@pytest.mark.parametrize("form", FORMS)
@pytest.mark.parametrize("case", sorted(all_cases()))
def test_edge_files(api, toks, case, form, tmp_path):
    texts = all_cases()[case]
    if case == "tiny_files" and form in ("gzip", "mixed"):
        texts = texts[:1000]  # single-member gzip of every file is the host's zlib speed, not the device's
    paths = write_files(tmp_path, case, texts, form)
    same_as_existing_paths(api, toks, paths, per_file=case != "tiny_files")


@pytest.fixture(scope="module")
def ctx():
    from gtars_b200 import ffi
    c = ffi.Context(0)
    yield c
    c.close()


@pytest.fixture(scope="module")
def index(ctx):
    """an ffi Bits index of overlapping peaks on NAMES: (index, names, unk id)"""
    from gtars_b200 import ffi
    rng = np.random.default_rng(31)
    per = 200
    s = rng.integers(0, 3400, len(NAMES) * per).astype(np.uint32)
    e = (s + rng.integers(20, 400, len(s))).astype(np.uint32)
    ix = ffi.Index(ctx, ffi.KIND_BITS, np.arange(len(NAMES) + 1, dtype=np.uint64) * per, s, e, np.arange(len(s), dtype=np.uint32))
    yield ix, NAMES, len(s)
    ix.close()


@gpu
def test_ffi_forms_and_no_files(index):
    """ffi.Index.tokenize_bed_files / _gz on the text and on the gzip members: file f's ids equal tokenize_bed on file f; zero
    files give the offsets [0] and no ids."""
    ix, names, unk = index
    texts = all_cases()["sorted_and_unsorted"] + all_cases()["no_final_newline"]
    fo = np.cumsum([0] + [len(t) for t in texts]).astype(np.uint64)
    members = [gzip.compress(t, mtime=0) for t in texts]
    mo = np.cumsum([0] + [len(m) for m in members]).astype(np.uint64)
    a = ix.tokenize_bed_files(b"".join(texts), fo, names, unk)
    b = ix.tokenize_bed_files_gz(b"".join(members), np.arange(len(texts) + 1), mo, names, unk)
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1]) and len(a[0]) == len(texts) + 1
    for f, t in enumerate(texts):
        assert a[1][int(a[0][f]):int(a[0][f + 1])].tolist() == ix.tokenize_bed(t, names, unk).tolist()
    off, ids = ix.tokenize_bed_files(b"", np.zeros(1, dtype=np.uint64), names, unk)
    assert off.tolist() == [0] and len(ids) == 0
    off, ids = ix.tokenize_bed_files_gz(b"", np.zeros(1, dtype=np.uint64), np.zeros(1, dtype=np.uint64), names, unk)
    assert off.tolist() == [0] and len(ids) == 0


@gpu
def test_forced_windows(api, toks, tmp_path, monkeypatch):
    """Windows of 1 byte to 64 KiB give the default window's ids, including file boundaries exactly on window cuts (every file of
    "aligned" is 64 bytes) and files whose last line has no '\\n'."""
    texts = all_cases()
    rng = np.random.default_rng(8)
    aligned = []
    for i in range(40):
        s = int(rng.integers(0, 3000))
        line = f"chr{1 + i % 3}\t{s:010d}\t{s + 50:010d}"            # 4 + 1 + 10 + 1 + 10 = 26 bytes
        aligned.append((line + "\n" + line[:-1] + "7" + "\t" + "x" * 9 + "\n").encode())
    assert all(len(t) == 64 for t in aligned)
    sets = {"aligned": aligned, "no_final_newline": texts["no_final_newline"], "comments_crlf": texts["comments_crlf"],
            "header_in_file_3": texts["header_in_file_3"], "sorted_and_unsorted": texts["sorted_and_unsorted"],
            "tiny": texts["tiny_files"][:300]}
    paths = {k: (write_files(tmp_path, k, v, "plain"), write_files(tmp_path, k, v, "bgzf")) for k, v in sets.items()}
    monkeypatch.delenv("GTGPU_INGEST_WINDOW", raising=False)
    want = {k: same_as_existing_paths(api, toks, p[0], per_file=False) for k, p in paths.items()}
    for w in ("1", "7", "64", "1024", "65536"):
        monkeypatch.setenv("GTGPU_INGEST_WINDOW", w)
        for k, (plain, bg) in paths.items():
            assert toks[0].encode_bed_files(plain) == want[k], (w, k)
            assert toks[0].encode_bed_files(bg) == want[k], (w, k)


def _file_line(msg):
    m = re.search(r"file (\d+), line (\d+)", msg)
    assert m, msg
    return int(m.group(1)), int(m.group(2))


@gpu
def test_errors_name_file_and_line(api, toks, index, tmp_path, monkeypatch):
    from gtars_b200 import ffi
    bits = toks[0]
    ix, names, unk = index
    rng = np.random.default_rng(9)
    good = [("\n".join(f"chr{1 + j % 2}\t{int(rng.integers(0, 3000))}\t3500" for j in range(300)) + "\n").encode() for _ in range(6)]
    good_paths = write_files(tmp_path, "good", good, "plain")
    want = bits.encode_bed_files(good_paths)
    assert want == [bits.encode_bed_file(p) for p in good_paths]

    def still_usable():
        assert bits.encode_bed_files(good_paths) == want

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
        for call in (lambda: ix.tokenize_bed_files(b"".join(bad), bfo, names, unk),
                     lambda: ix.tokenize_bed_files_gz(b"".join(members), np.arange(len(bad) + 1), mo, names, unk)):
            with pytest.raises(ffi.GtarsGpuError) as e:
                call()
            assert e.value.code == 1 and _file_line(str(e.value)) == (k, j), str(e.value)
            still_usable()
        for form in ("plain", "gzip", "mixed"):
            paths = write_files(tmp_path, f"bad{k}", bad, form)
            with pytest.raises(api.GtarsError) as e:
                bits.encode_bed_files(paths)
            assert paths[k] in str(e.value) and f"line {j}" in str(e.value), str(e.value)
            still_usable()
        monkeypatch.delenv("GTGPU_INGEST_WINDOW", raising=False)
    for empty in (b"", b"# only\n#comments\ntrack x\n", b"chrom\tstart\tend\n"):
        texts = good[:2] + [empty] + good[2:]
        efo = np.cumsum([0] + [len(t) for t in texts]).astype(np.uint64)
        with pytest.raises(ffi.GtarsGpuError) as e:
            ix.tokenize_bed_files(b"".join(texts), efo, names, unk)
        assert e.value.code == 1 and "file 2: " in str(e.value) and "0 regions" in str(e.value)
        for form in ("plain", "gzip"):
            paths = write_files(tmp_path, "empty", texts, form)
            with pytest.raises(api.GtarsError) as e:
                bits.encode_bed_files(paths)
            assert paths[2] in str(e.value) and "0 regions" in str(e.value)
            still_usable()
    # a last line ending in '\r' without '\n' is malformed, as the device parser has it (test_final_cr_follows_the_device_parser)
    t = b"chr1\t1\t10\nchr1\t5\t20\r"
    for texts in ([t], [b"chr2\t1\t5\n", t], [t, b"chr2\t1\t5\n"]):
        fo = np.cumsum([0] + [len(x) for x in texts]).astype(np.uint64)
        with pytest.raises(ffi.GtarsGpuError) as e:
            ix.tokenize_bed_files(b"".join(texts), fo, names, unk)
        assert _file_line(str(e.value)) == (texts.index(t), 2)
        still_usable()


def c2_batch(n_files, per_file, seed=0):
    """C2-shaped query files (synth) against a 1e6-peak universe: (index args, chr / start / end, file offsets, unk id)"""
    from gtars_b200 import synth
    u = synth.make_universe(1_000_000)
    q = synth.make_query_files(u, n_files, per_file, seed=0x5EED0002 + seed)
    ix_args = (u["chrom_offsets"].numpy().astype(np.uint64), *(u[k].numpy().view(np.uint32) for k in ("g_start", "g_end", "g_val")))
    return ix_args, [q[k].numpy().view(np.uint32) for k in ("chr", "start", "end")], u["unk_id"]


def shuffled_within_files(c, s, e, per_file, rng):
    n_files = len(c) // per_file
    perm = (np.argsort(rng.random((n_files, per_file)), axis=1) + np.arange(n_files)[:, None] * per_file).ravel()
    return c[perm], s[perm], e[perm]


def file_sorted(c, s, e, per_file):
    """RegionSet::sort per file: stable by (chromosome string, start)"""
    from gtars_b200 import synth
    rank = synth.lex_rank("cpu").numpy()[c.astype(np.int64)]
    order = np.lexsort((s, rank, np.arange(len(c)) // per_file))
    return c[order], s[order], e[order]


def check_against_arrays(ix, c, s, e, per_file, unk):
    """tokenize_bed_files over the records as BED text == tokenize_files over the per-file sorted arrays"""
    from gtars_b200 import synth
    n_files = len(c) // per_file
    text = bed_text(c.astype(np.int64), s, e)
    fo = np.concatenate([[0], np.flatnonzero(text == 10)[per_file - 1::per_file] + 1]).astype(np.uint64)
    got = ix.tokenize_bed_files(text, fo, synth.CHROM_NAMES, unk)
    del text
    want = ix.tokenize_files(np.arange(n_files + 1, dtype=np.uint64) * np.uint64(per_file), *file_sorted(c, s, e, per_file), unk)
    assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1])
    return got


@gpu
def test_file_pass_when_file_and_rank_do_not_fit_one_key(index):
    """2 100 small unsorted files: with the index's names the file index is folded into the rank key (6 + 12 bits); with 2^20 more
    names in the table (21 + 12 bits > 32) it takes a radix pass of its own.  Both equal gtgpu_tokenize_files on the files
    stable-sorted by (name string, start) on the host."""
    ix, names, unk = index
    rng = np.random.default_rng(41)
    n_files, per = 2100, 6
    used = names + ["chrNowhere"]
    c = rng.integers(0, len(used), n_files * per)
    s = rng.integers(0, 3000, n_files * per).astype(np.uint32) // 50 * 50     # ties on (name, start)
    e = (s + rng.integers(1, 500, len(s))).astype(np.uint32)
    texts = ["".join(f"{used[c[k]]}\t{s[k]}\t{e[k]}\n" for k in range(f * per, (f + 1) * per)).encode() for f in range(n_files)]
    fo = np.cumsum([0] + [len(t) for t in texts]).astype(np.uint64)
    by_string = {n: r for r, n in enumerate(sorted(used))}
    order = np.lexsort((s, [by_string[used[x]] for x in c], np.arange(len(c)) // per))
    ids = np.array([i if i < len(names) else 0xFFFFFFFF for i in c], dtype=np.uint32)
    want = ix.tokenize_files(np.arange(n_files + 1, dtype=np.uint64) * per, ids[order], s[order], e[order], unk)
    for table in (names, names + [f"pad{i:07d}" for i in range(1 << 20)]):
        got = ix.tokenize_bed_files(b"".join(texts), fo, table, unk)
        assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1]), len(table)


@gpu
def test_c2_shape_reduced_sorted_and_shuffled():
    """200 files x 1e5 regions from synth as BED text == gtgpu_tokenize_files on the generated arrays; shuffled within every file,
    the device sorts them back to the same answer."""
    from gtars_b200 import ffi
    per = 100_000
    ix_args, (c, s, e), unk = c2_batch(200, per)
    ctx = ffi.Context(0)
    ix = ffi.Index(ctx, ffi.KIND_BITS, *ix_args)
    sorted_res = check_against_arrays(ix, c, s, e, per, unk)
    shuf = check_against_arrays(ix, *shuffled_within_files(c, s, e, per, np.random.default_rng(1)), per, unk)
    assert np.array_equal(sorted_res[0], shuf[0])                   # same hits per file, ties on (name, start) aside
    ix.close()
    ctx.close()


@gpu
def test_text_past_4_gib():
    """18 files of 1e7 regions (more than 4.4 GB of text) in the default 2 GiB windows, every other file shuffled: equal to
    gtgpu_tokenize_files on the per-file sorted arrays."""
    from gtars_b200 import ffi, synth
    per, reps = 10_000_000, 18
    ix_args, (c, s, e), unk = c2_batch(1, per, seed=5)
    shuf = shuffled_within_files(c, s, e, per, np.random.default_rng(2))
    chunks = [bed_text(c.astype(np.int64), s, e), bed_text(shuf[0].astype(np.int64), shuf[1], shuf[2])]
    text = np.concatenate([chunks[f % 2] for f in range(reps)])
    assert text.nbytes > 4.4e9
    fo = np.cumsum([0] + [chunks[f % 2].nbytes for f in range(reps)]).astype(np.uint64)
    del chunks
    ctx = ffi.Context(0)
    ix = ffi.Index(ctx, ffi.KIND_BITS, *ix_args)
    got = ix.tokenize_bed_files(text, fo, synth.CHROM_NAMES, unk)
    del text
    resorted = file_sorted(*shuf, per)
    want = ix.tokenize_files(np.arange(reps + 1, dtype=np.uint64) * np.uint64(per),
                             *(np.concatenate([(x, y)[f % 2] for f in range(reps)]) for x, y in zip((c, s, e), resorted)), unk)
    assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1])
    ix.close()
    ctx.close()


@gpu
def test_multi_device_context_equals_single():
    from gtars_b200 import ffi, synth
    if ffi.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    per = 20_000
    ix_args, (c, s, e), unk = c2_batch(37, per, seed=3)
    c, s, e = shuffled_within_files(c, s, e, per, np.random.default_rng(4))
    text = bed_text(c.astype(np.int64), s, e)
    fo = np.concatenate([[0], np.flatnonzero(text == 10)[per - 1::per] + 1]).astype(np.uint64)
    res = []
    for ctx in (ffi.Context(0), ffi.Context(devices=[0, 1])):
        ix = ffi.Index(ctx, ffi.KIND_BITS, *ix_args)
        res.append(ix.tokenize_bed_files(text, fo, synth.CHROM_NAMES, unk))
        ix.close()
        ctx.close()
    assert np.array_equal(res[0][0], res[1][0]) and np.array_equal(res[0][1], res[1][1])


def test_bench_script_writes_its_corpus(tmp_path):
    """profiles/tokenize_bed_files_bench.py at a tiny size, as far as it goes without a device: arguments, corpus, sizes."""
    r = subprocess.run([sys.executable, os.path.join(ROOT, "profiles", "tokenize_bed_files_bench.py"), "--files", "3", "--regions",
                        "500", "--universe", "5000", "--write-only"], capture_output=True, text=True, check=True,
                       env=dict(os.environ, TMPDIR=str(tmp_path)))
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["workload"] == "write_files" and line["files"] == 3
    assert line["file_bytes"]["plain"] == line["file_bytes"]["unsorted"] > line["file_bytes"]["gzip"] > 0
    assert os.listdir(tmp_path) == []                                # the corpus directory is removed at the end


@gpu
def test_bench_script_on_the_gpu(tmp_path):
    """The three timings at a tiny size, equal answers, with the card's name and power limit."""
    r = subprocess.run([sys.executable, os.path.join(ROOT, "profiles", "tokenize_bed_files_bench.py"), "--files", "4", "--regions",
                        "2000", "--universe", "20000", "--reps", "1"], capture_output=True, text=True, check=True,
                       env=dict(os.environ, TMPDIR=str(tmp_path)))
    lines = [json.loads(x) for x in r.stdout.strip().splitlines()]
    timed = [x for x in lines if x["workload"] == "tokenize_bed_files"]
    assert sorted({x["arm"] for x in timed}) == ["encode_bed_file_per_file", "encode_bed_files", "host_parse_encode_batch"]
    assert {x["format"] for x in timed} == {"plain", "gzip", "unsorted"}
    assert all(x["equal"] and x["gpu"] and x["power_limit"] and x["wall_s"] > 0 for x in timed)
