"""region_scoring_from_fragments / barcode_scoring_from_fragments with device_parse=True (gtgpu_score_matrix_text / _gz,
gtgpu_score_barcodes_text / _gz): the fragment file's text or BGZF bytes parsed on the device, in windows of
GTGPU_INGEST_WINDOW bytes, against the host parser, the oracle and the array entry points."""
import gzip
import os
import re
import struct
import zlib

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

CONSENSUS = ("chr1\t0\t8\n"          # reached by the wrapped ATAC arithmetic of end < 5
             "chr1\t100\t200\nchr1\t150\t400\nchr1\t1000\t1100\nchr1\t5000\t9000\n"
             "chr2\t50\t80\nchr2\t300\t310\nchrX\t10\t4000\nchrX\t4294967290\t4294967295\n")


@pytest.fixture(scope="module")
def api():
    from gtars_b200 import api as a
    a.device(0)
    return a


@pytest.fixture(scope="module")
def cons(api, tmp_path_factory):
    p = str(tmp_path_factory.mktemp("cons") / "consensus.bed")
    with open(p, "w") as f:
        f.write(CONSENSUS)
    return p, api.ConsensusSet(p)


def bgzf(data: bytes, block=None) -> bytes:
    """BGZF as bgzip writes it (independent members with the 'BC' extra field + the empty EOF block); small blocks so that
    even short texts have >= 16 members and take the device inflater."""
    block = block or max(64, -(-len(data) // 20))
    out = []
    for ch in [data[i:i + block] for i in range(0, len(data), block)] + [b""]:
        co = zlib.compressobj(6, zlib.DEFLATED, -15)
        body = co.compress(ch) + co.flush()
        out.append(b"\x1f\x8b\x08\x04" + b"\0" * 4 + b"\x00\xff" + struct.pack("<H", 6) + b"BC" + struct.pack("<HH", 2, 12 + 6 + len(body) + 8 - 1)
                   + body + struct.pack("<II", zlib.crc32(ch), len(ch)))
    return b"".join(out)


def variants(d, name, text: bytes):
    """The same text as plain, BGZF and single-member gzip files."""
    paths = [str(d / f"{name}.tsv"), str(d / f"{name}.bgzf.tsv.gz"), str(d / f"{name}.one.tsv.gz")]
    for p, data in zip(paths, (text, bgzf(text), gzip.compress(text, mtime=0))):
        with open(p, "wb") as f:
            f.write(data)
    return paths


def random_lines(rng, n, names=("chr1", "chr2", "chrX", "chr9"), n_bc=40, bc_prefix="BC"):
    out = []
    for _ in range(n):
        c = names[int(rng.integers(0, len(names)))]
        s = int(rng.integers(0, 6000))
        out.append(f"{c}\t{s}\t{s + int(rng.integers(1, 600))}\t{bc_prefix}{int(rng.integers(0, n_bc))}\t{int(rng.integers(1, 9))}")
    return out


def cases():
    rng = np.random.default_rng(11)
    lines = random_lines(rng, 300)
    c = {}
    c["comments"] = "# header line\n#another\n" + "\n".join(lines[:150] + ["# in the middle", "#"] + lines[150:]) + "\n"
    ws = []
    for i, l in enumerate(lines):
        f = l.split("\t")
        sep = ["\t", " ", "  ", " \t", "\t\t"][i % 5]
        ws.append((" " if i % 7 == 0 else "") + sep.join(f) + (" \t" if i % 3 == 0 else ""))
    c["whitespace_crlf"] = "\r\n".join(ws) + "\r\n"
    c["extra_columns"] = "\n".join(l + "\textra\t+\t0.5" for l in lines) + "\n"
    c["unknown_chroms"] = "\n".join(lines[:100] + ["chrUn\t10\t20\tGHOST\t1", "chr9\t100\t200\tGHOST\t2", "chrUn\t1\t2\tBC1\t1"]
                                    + lines[100:]) + "\n"
    c["end_below_5"] = "\n".join(lines[:50] + ["chr1\t0\t3\tW1\t1", "chr1\t2\t4\tW2\t1", "chr1\t0\t0\tW1\t1", "chrX\t4294967291\t4294967295\tW3\t1",
                                               "chr1\t4294967295\t4294967295\tW4\t1"] + lines[50:]) + "\n"
    c["no_trailing_newline"] = "\n".join(lines)
    c["no_trailing_newline_cr"] = "\n".join(lines) + "\r"
    c["empty"] = ""
    c["comments_only"] = "# nothing\n#\n# here\n"
    return {k: v.encode() for k, v in c.items()}


def same_matrix(api, cons_path, cs, files):
    from oracle import oracle as orc
    for mode in (api.SCORING_ATAC, api.SCORING_CHIP):
        dev = api.region_scoring_from_fragments(files, cs, mode, device_parse=True)
        host = api.region_scoring_from_fragments(files, cs, mode)
        assert np.array_equal(dev, host), (files, mode)
        assert np.array_equal(dev, orc.region_scoring_files(cons_path, files, mode)), (files, mode)


def same_barcodes(api, cons_path, cs, path, check_oracle=True):
    from oracle import oracle as orc
    dev = api.barcode_scoring_from_fragments(path, cs, device_parse=True)
    host = api.barcode_scoring_from_fragments(path, cs)
    assert dev == host and list(dev) == list(host), path          # key set and first-appearance order
    if check_oracle:
        assert dev == orc.barcode_scoring_file(cons_path, path), path
    return dev


def test_kat_k10_through_device_parse(api, golden, fixture_dir):
    """K10 (gtars-scoring/src/fragment_scoring.rs:180-210) with device_parse=True: the golden ATAC matrix, the Chip matrix
    of the host path, and the per-barcode counts of fragments1 including the oracle's key set and order."""
    from oracle import oracle as orc
    k = golden[1]["K10_scoring"]
    cons_path = os.path.join(fixture_dir, k["consensus"])
    cs = api.ConsensusSet(cons_path)
    files = [os.path.join(fixture_dir, f) for f in k["fragment_files"]]
    m = api.region_scoring_from_fragments(files, cs, api.SCORING_ATAC, device_parse=True)
    assert m.tolist() == k["matrix"]
    assert np.array_equal(m, api.region_scoring_from_fragments(files, cs, api.SCORING_ATAC))
    chip = api.region_scoring_from_fragments(files, cs, api.SCORING_CHIP, device_parse=True)
    assert np.array_equal(chip, api.region_scoring_from_fragments(files, cs, api.SCORING_CHIP))
    got = api.barcode_scoring_from_fragments(files[0], cs, device_parse=True)
    want = orc.barcode_scoring_file(cons_path, files[0])
    assert got == want and list(got) == list(want)
    assert got == api.barcode_scoring_from_fragments(files[0], cs)


@pytest.mark.parametrize("case", sorted(cases()))
def test_generated_files_device_host_oracle(api, cons, tmp_path, case):
    cons_path, cs = cons
    for p in variants(tmp_path, case, cases()[case]):
        same_matrix(api, cons_path, cs, [p])
        got = same_barcodes(api, cons_path, cs, p)
        if case == "unknown_chroms":
            assert "GHOST" not in got and "BC1" in got


def test_several_files_one_empty(api, cons, tmp_path):
    cons_path, cs = cons
    c = cases()
    files = [variants(tmp_path, "a", c["comments"])[0], variants(tmp_path, "e", c["empty"])[1],
             variants(tmp_path, "b", c["whitespace_crlf"])[1], variants(tmp_path, "o", c["comments_only"])[2],
             variants(tmp_path, "u", c["unknown_chroms"])[2]]
    same_matrix(api, cons_path, cs, files)
    m = api.region_scoring_from_fragments(files, cs, api.SCORING_ATAC, device_parse=True)
    assert m[1].sum() == 0 and m[3].sum() == 0 and m[0].sum() > 0


def _line_of(msg):
    m = re.search(r"at line (\d+)\b", msg)
    assert m, msg
    return int(m.group(1))


MALFORMED = {
    "four_fields": "chr1\t100\t200\tBC",
    "start_x": "chr1\tx\t200\tBC\t1", "start_neg": "chr1\t-1\t200\tBC\t1", "start_big": "chr1\t4294967296\t200\tBC\t1",
    "end_x": "chr1\t100\tx\tBC\t1", "end_neg": "chr1\t100\t-1\tBC\t1", "end_big": "chr1\t100\t4294967296\tBC\t1",
    "support_x": "chr1\t100\t200\tBC\tx", "support_neg": "chr1\t100\t200\tBC\t-1", "support_big": "chr1\t100\t200\tBC\t4294967296",
}


@pytest.mark.parametrize("bad", sorted(MALFORMED))
def test_malformed_line_is_reported_like_the_host(api, cons, tmp_path, bad):
    _, cs = cons
    rng = np.random.default_rng(5)
    good = random_lines(rng, 60)
    text = ("#c\n" + "\n".join(good[:37] + [MALFORMED[bad]] + good[37:]) + "\n").encode()
    for p in variants(tmp_path, bad, text):
        with pytest.raises(api.GtarsError) as host:
            api.region_scoring_from_fragments([p], cs)
        for call in (lambda: api.region_scoring_from_fragments([p], cs, device_parse=True),
                     lambda: api.barcode_scoring_from_fragments(p, cs, device_parse=True)):
            with pytest.raises(api.GtarsError) as dev:
                call()
            assert _line_of(str(dev.value)) == _line_of(str(host.value)) == 38 and p in str(dev.value), (str(dev.value), str(host.value))


def test_bad_line_in_the_second_of_three_files(api, cons, tmp_path):
    _, cs = cons
    rng = np.random.default_rng(6)
    ok = ("\n".join(random_lines(rng, 50)) + "\n").encode()
    bad = ("\n".join(random_lines(rng, 20) + ["chr1\t5\t9\tBC\t1.5"] + random_lines(rng, 5)) + "\n").encode()
    files = [variants(tmp_path, "f0", ok)[0], variants(tmp_path, "f1", bad)[1], variants(tmp_path, "f2", ok)[2]]
    with pytest.raises(api.GtarsError) as host:
        api.region_scoring_from_fragments(files, cs)
    with pytest.raises(api.GtarsError) as dev:
        api.region_scoring_from_fragments(files, cs, device_parse=True)
    assert _line_of(str(dev.value)) == _line_of(str(host.value)) == 20
    assert files[1] in str(dev.value) and files[0] not in str(dev.value) and files[2] not in str(dev.value)


def _window_text(rng):
    """~120 KB of fragments with '\\r\\n' and '#' lines throughout, barcodes that first appear late, and three prefixes that put
    the 1 KiB boundary (byte 1023) on a '\\n', inside a '\\r\\n' and inside a '#' line."""
    lines = []
    for i in range(2500):
        l = random_lines(rng, 1, n_bc=30 + i // 10)[0]                    # the barcode alphabet grows: new barcodes in late windows
        lines.append(l + ("\r" if i % 3 == 0 else ""))
        if i % 97 == 0:
            lines.append("# comment " + "x" * int(rng.integers(0, 300)))
    return lines


def _pad_to(first, byte_at_1023, crlf):
    """A valid first line padded (sixth column) so that byte 1023 of the text is `byte_at_1023`."""
    end = "\r\n" if crlf else "\n"
    pad = 1024 - len(first) - 1 - len(end) + (1 if byte_at_1023 == "\r" else 0)
    return first + "\t" + "p" * pad + end


def test_windows_give_the_single_window_result(api, cons, tmp_path, monkeypatch):
    cons_path, cs = cons
    rng = np.random.default_rng(21)
    body = "\n".join(_window_text(rng)) + "\n"
    head = "chr1\t120\t130\tFIRST\t1"
    texts = {"nl": _pad_to(head, "\n", False) + body, "crlf": _pad_to(head, "\r", True) + body,
             "comment": head + "\n" + "#" + "c" * 2000 + "\n" + body}
    assert texts["nl"][1023] == "\n" and texts["crlf"][1023] == "\r" and texts["crlf"][1024] == "\n"
    assert texts["comment"].index("#") < 1023 < texts["comment"].index("\n", texts["comment"].index("#"))
    paths = {k: variants(tmp_path, k, v.encode())[:2] for k, v in texts.items()}
    monkeypatch.delenv("GTGPU_INGEST_WINDOW", raising=False)
    want = {k: (api.region_scoring_from_fragments(ps, cs, api.SCORING_ATAC, device_parse=True),
                [api.barcode_scoring_from_fragments(p, cs, device_parse=True) for p in ps]) for k, ps in paths.items()}
    for k, ps in paths.items():
        assert np.array_equal(want[k][0], api.region_scoring_from_fragments(ps, cs, api.SCORING_ATAC))
        assert want[k][1][0] == api.barcode_scoring_from_fragments(ps[0], cs)
    for w in ("1024", "4096", "65536", "1"):
        monkeypatch.setenv("GTGPU_INGEST_WINDOW", w)
        for k, ps in paths.items():
            assert np.array_equal(api.region_scoring_from_fragments(ps, cs, api.SCORING_ATAC, device_parse=True), want[k][0]), (w, k)
            for p, b in zip(ps, want[k][1]):
                got = api.barcode_scoring_from_fragments(p, cs, device_parse=True)
                assert got == b and list(got) == list(b), (w, k, p)


def test_bad_line_in_a_late_window(api, cons, tmp_path, monkeypatch):
    _, cs = cons
    rng = np.random.default_rng(22)
    lines = _window_text(rng)
    lines.insert(len(lines) - 40, "chr2\t1\t2\tLATE")
    ps = variants(tmp_path, "late", ("\n".join(lines) + "\n").encode())
    with pytest.raises(api.GtarsError) as host:
        api.region_scoring_from_fragments([ps[0]], cs)
    want = _line_of(str(host.value))
    assert want == len(lines) - 41
    monkeypatch.setenv("GTGPU_INGEST_WINDOW", "1024")
    for p in ps:
        for call in (lambda: api.region_scoring_from_fragments([p], cs, device_parse=True),
                     lambda: api.barcode_scoring_from_fragments(p, cs, device_parse=True)):
            with pytest.raises(api.GtarsError) as dev:
                call()
            assert _line_of(str(dev.value)) == want and p in str(dev.value)


# ---- past 4 GiB of text ------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def universe_index():
    from gtars_b200 import ffi, synth
    u = synth.make_universe(200_000)
    offs = u["chrom_offsets"].numpy().astype(np.uint64)
    s, e, v = (u[k].numpy().view(np.uint32) for k in ("g_start", "g_end", "g_val"))
    ctx = ffi.Context(0)
    ix = ffi.Index(ctx, ffi.KIND_BITS, offs, s, e, v)
    yield ix, int(u["n"])
    ix.close()
    ctx.close()


def test_text_past_4_gib(universe_index):
    """One plain text of > 4 GiB (1.1e8 fragments) in the default 2 GiB windows == gtgpu_score_matrix on the arrays."""
    from gtars_b200 import ffi, synth
    ix, n_cols = universe_index
    n, chunk, L = 110_000_000, 10_000_000, synth.FRAGMENT_LINE
    text = np.empty(n * L, dtype=np.uint8)
    cols = [np.empty(n, dtype=np.uint32) for _ in range(3)]
    for a in range(0, n, chunk):
        c, s, e, b = synth.make_fragment_arrays(min(chunk, n - a), 1000 + a // chunk, 10**6)
        text[a * L:(a + len(s)) * L] = synth.fragment_text(c, s, e, b)
        for dst, src in zip(cols, (c, s, e)):
            dst[a:a + len(s)] = src
    assert text.nbytes > 4 << 30
    fo = np.array([0, n], dtype=np.uint64)
    for mode in (ffi.SCORE_ATAC, ffi.SCORE_CHIP):
        want = ix.score_matrix(fo, *cols, mode, n_cols)[0]
        assert want.sum() > 0
        assert np.array_equal(ix.score_matrix_text(text, synth.CHROM_NAMES, mode, n_cols), want), mode


def test_barcodes_at_scale_and_oracle_slice(api, universe_index, tmp_path):
    """3e7 fragments: the barcode CSR == gtgpu_score_barcodes with ids in first-appearance order; a slice written as a file
    and read through the API == the oracle."""
    from gtars_b200 import ffi, synth
    from oracle import oracle as orc
    ix, n_cols = universe_index
    c, s, e, b = synth.make_fragment_arrays(30_000_000, 77, 400_000)
    text = synth.fragment_text(c, s, e, b)
    _, first = np.unique(b, return_index=True)
    order = np.argsort(first, kind="stable")
    dense = np.empty(order.size, dtype=np.uint32)
    dense[np.unique(b)[order]] = np.arange(order.size, dtype=np.uint32)
    want_off, want_pk, want_ct = ix.score_barcodes(c, s, e, dense[b], order.size)
    names, off, pk, ct = ix.score_barcodes_text(text, synth.CHROM_NAMES)
    assert names == ["BC%07d" % x for x in np.unique(b)[order]]
    assert np.array_equal(off, want_off) and np.array_equal(pk, want_pk) and np.array_equal(ct, want_ct)
    gz = bgzf(text[:4_000_000].tobytes(), block=60_000)
    names2, off2, pk2, ct2 = ix.score_barcodes_text(gz, synth.CHROM_NAMES, gz_member_offsets=ffi.gzip_members(gz))
    n2, o2, p2, c2 = ix.score_barcodes_text(text[:4_000_000], synth.CHROM_NAMES)
    assert names2 == n2 and np.array_equal(off2, o2) and np.array_equal(pk2, p2) and np.array_equal(ct2, c2)
    # the slice through the host layer vs the oracle (a consensus file of the universe's first 20 000 peaks, sorted)
    cons_path, frag_path = str(tmp_path / "cons.bed"), str(tmp_path / "slice.tsv")
    u = synth.make_universe(20_000)
    uc, us, ue = (u[k].numpy() for k in ("chr", "start", "end"))
    with open(cons_path, "w") as f:
        f.write("".join(f"{synth.CHROM_NAMES[x]}\t{y}\t{z}\n" for x, y, z in zip(uc, us, ue)))
    with open(frag_path, "wb") as f:
        f.write(text[:200_000 * synth.FRAGMENT_LINE].tobytes())
    got = api.barcode_scoring_from_fragments(frag_path, api.ConsensusSet(cons_path), device_parse=True)
    assert got == orc.barcode_scoring_file(cons_path, frag_path) and len(got) > 1000


def test_multi_device_context_equals_single(universe_index):
    from gtars_b200 import ffi, synth
    if ffi.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    ix1, n_cols = universe_index
    u = synth.make_universe(200_000)
    offs = u["chrom_offsets"].numpy().astype(np.uint64)
    s, e, v = (u[k].numpy().view(np.uint32) for k in ("g_start", "g_end", "g_val"))
    ctx = ffi.Context(devices=[0, 1])
    ixm = ffi.Index(ctx, ffi.KIND_BITS, offs, s, e, v)
    c, fs, fe, b = synth.make_fragment_arrays(2_000_000, 5, 5000)
    text = synth.fragment_text(c, fs, fe, b)
    for mode in (ffi.SCORE_ATAC, ffi.SCORE_CHIP):
        assert np.array_equal(ixm.score_matrix_text(text, synth.CHROM_NAMES, mode, n_cols), ix1.score_matrix_text(text, synth.CHROM_NAMES, mode, n_cols))
    a, bb = ixm.score_barcodes_text(text, synth.CHROM_NAMES), ix1.score_barcodes_text(text, synth.CHROM_NAMES)
    assert a[0] == bb[0] and all(np.array_equal(x, y) for x, y in zip(a[1:], bb[1:]))
    ixm.close()
    ctx.close()
