"""tokenize_fragment_file from a fragment file's text or gzip bytes of any size (gtgpu_tokenize_fragments_file / _gz, and
api.tokenize_fragment_file with device_parse=True), parsed on the device in windows of GTGPU_INGEST_WINDOW bytes, against
gtgpu_tokenize_fragments_text, the host parser, the oracle, the D3 known answer and the array entry point."""
import ctypes as C
import gzip
import os
import re
import struct
import zlib

import numpy as np
import pytest

from tests.test_gpu_score_text import _pad_to, _window_text, cases, variants

pytestmark = pytest.mark.gpu

UNIVERSE = ("chr1\t0\t8\nchr1\t100\t200\nchr1\t150\t400\nchr1\t1000\t1100\nchr1\t5000\t9000\n"
            "chr2\t50\t80\nchr2\t300\t310\nchrX\t10\t4000\nchrX\t4294967290\t4294967295\n")


@pytest.fixture(scope="module")
def api():
    from gtars_b200 import api as a
    a.device(0)
    return a


@pytest.fixture(scope="module")
def tok(api, tmp_path_factory):
    p = str(tmp_path_factory.mktemp("uni") / "universe.bed")
    with open(p, "w") as f:
        f.write(UNIVERSE)
    return p, api.Tokenizer(p)


@pytest.fixture(scope="module")
def small_index():
    """An ffi index over the same universe, chromosome names in the order the text forms take them."""
    from gtars_b200 import ffi
    names = ["chr1", "chr2", "chrX"]
    rows = [l.split("\t") for l in UNIVERSE.splitlines()]
    offs = np.array([0, 5, 7, 9], dtype=np.uint64)
    s, e = (np.array([int(r[k]) for r in rows], dtype=np.uint32) for k in (1, 2))
    ctx = ffi.Context(0)
    ix = ffi.Index(ctx, ffi.KIND_BITS, offs, s, e, np.arange(len(rows), dtype=np.uint32))
    yield ix, names, len(rows)
    ix.close()
    ctx.close()


@pytest.fixture(scope="module")
def universe_index():
    from gtars_b200 import ffi, synth
    u = synth.make_universe(200_000)
    offs = u["chrom_offsets"].numpy().astype(np.uint64)
    s, e, v = (u[k].numpy().view(np.uint32) for k in ("g_start", "g_end", "g_val"))
    ctx = ffi.Context(0)
    ix = ffi.Index(ctx, ffi.KIND_BITS, offs, s, e, v)
    yield ix, u
    ix.close()
    ctx.close()


def bgzf_fast(data, block=65_280) -> bytes:
    """BGZF at zlib level 1 (large texts), blocks as bgzip writes them plus the empty EOF block."""
    mv = memoryview(data)
    out = []
    for a in list(range(0, len(mv), block)) + [len(mv)]:
        ch = bytes(mv[a:a + block])
        co = zlib.compressobj(1, zlib.DEFLATED, -15)
        body = co.compress(ch) + co.flush()
        out.append(b"\x1f\x8b\x08\x04" + b"\0" * 4 + b"\x00\xff" + struct.pack("<H", 6) + b"BC" + struct.pack("<HH", 2, 12 + 6 + len(body) + 8 - 1)
                   + body + struct.pack("<II", zlib.crc32(ch), len(ch)))
    return b"".join(out)


def file_form(ix, names, unk, text):
    """gtgpu_tokenize_fragments_file on the text, and _gz on its BGZF form: both equal, returned once."""
    from gtars_b200 import ffi
    got = ix.tokenize_fragments_file(text, names, unk)
    gz = bgzf_fast(bytes(text), block=max(64, -(-len(text) // 20)))
    got_gz = ix.tokenize_fragments_file(gz, names, unk, gz_member_offsets=ffi.gzip_members(gz))
    assert got_gz[0] == got[0] and np.array_equal(got_gz[1], got[1]) and np.array_equal(got_gz[2], got[2])
    return got


def same_as_text_form(ix, names, unk, text):
    b, o, i = file_form(ix, names, unk, text)
    tb, to, ti = ix.tokenize_fragments_text(text, names, unk)
    assert b == tb and np.array_equal(o, to) and np.array_equal(i, ti)
    assert len(o) == len(b) + 1 and o[-1] == len(i)
    return b, o, i


def same_through_api(api, tok, path):
    from oracle import oracle as orc
    uni, t = tok
    dev = api.tokenize_fragment_file(path, t, device_parse=True)
    host = api.tokenize_fragment_file(path, t)
    assert dev == host and list(dev) == list(host), path           # same lists, same first-appearance order
    assert dev == orc.Tokenizer(uni).tokenize_fragment_file(path), path
    return dev


def _line_of(msg):
    m = re.search(r"at line:? (\d+)\b", msg)
    assert m, msg
    return int(m.group(1))


def test_kat_d3(api, golden, fixture_dir, tmp_path):
    """D3 (the reference's fragment fixture) as plain text, BGZF and single-member gzip."""
    d3 = golden[1]["D_derived"]["D3"]
    t = api.Tokenizer(os.path.join(fixture_dir, d3["universe"]))
    src = os.path.join(fixture_dir, d3["fragments"])
    with open(src, "rb") as f:
        raw = f.read()
    text = gzip.decompress(raw) if src.endswith(".gz") else raw
    for p in variants(tmp_path, "d3", text):
        assert api.tokenize_fragment_file(p, t, device_parse=True) == d3["expect"], p


@pytest.mark.parametrize("case", sorted(cases()))
def test_edge_cases(api, tok, small_index, tmp_path, case):
    ix, names, unk = small_index
    text = cases()[case]
    b, _, i = same_as_text_form(ix, names, unk, text)
    for p in variants(tmp_path, case, text):
        got = same_through_api(api, tok, p)
        if case == "unknown_chroms":
            assert got["GHOST"] and "GHOST" in b           # a barcode seen only on unknown chromosomes is kept
        if case in ("empty", "comments_only"):
            assert got == {} and b == [] and len(i) == 0


def test_windows_give_the_single_window_result(api, tok, small_index, tmp_path, monkeypatch):
    """Windows of 1 byte to 64 KiB, cut at a '\\n', at the '\\r' of a '\\r\\n' and inside a long '#' line; barcodes first appear
    in late windows and reappear across windows."""
    ix, names, unk = small_index
    rng = np.random.default_rng(41)
    body = "\n".join(_window_text(rng)) + "\n"
    head = "chr1\t120\t130\tFIRST\t1"
    texts = {"nl": _pad_to(head, "\n", False) + body, "crlf": _pad_to(head, "\r", True) + body,
             "comment": head + "\n" + "#" + "c" * 2000 + "\n" + body}
    assert texts["nl"][1023] == "\n" and texts["crlf"][1023] == "\r" and texts["crlf"][1024] == "\n"
    texts = {k: v.encode() for k, v in texts.items()}
    paths = {k: variants(tmp_path, k, v)[:2] for k, v in texts.items()}
    monkeypatch.delenv("GTGPU_INGEST_WINDOW", raising=False)
    want = {k: same_as_text_form(ix, names, unk, v) for k, v in texts.items()}
    want_api = {k: [same_through_api(api, tok, p) for p in ps] for k, ps in paths.items()}
    late = {b for b in want["nl"][0] if body.encode().find(b.encode() + b"\t") > len(body) // 2}
    assert len(late) > 10                                            # barcodes whose first appearance lies in a late window
    for w in ("1", "1024", "4096", "65536"):
        monkeypatch.setenv("GTGPU_INGEST_WINDOW", w)
        for k, v in texts.items():
            got = same_as_text_form(ix, names, unk, v)
            assert got[0] == want[k][0] and all(np.array_equal(x, y) for x, y in zip(got[1:], want[k][1:])), (w, k)
            for p, d in zip(paths[k], want_api[k]):
                got_api = api.tokenize_fragment_file(p, tok[1], device_parse=True)
                assert got_api == d and list(got_api) == list(d), (w, k, p)


def test_bad_line_in_a_late_window(api, tok, small_index, tmp_path, monkeypatch):
    ix, names, unk = small_index
    rng = np.random.default_rng(42)
    lines = _window_text(rng)
    good = ("\n".join(lines) + "\n").encode()
    lines.insert(len(lines) - 40, "chr2\t1\t2\tLATE")
    bad = ("\n".join(lines) + "\n").encode()
    ps = variants(tmp_path, "late", bad)
    with pytest.raises(api.GtarsError) as host:
        api.tokenize_fragment_file(ps[0], tok[1])
    want = _line_of(str(host.value))
    assert want == len(lines) - 41
    monkeypatch.setenv("GTGPU_INGEST_WINDOW", "1024")
    for p in ps:
        with pytest.raises(api.GtarsError) as dev:
            api.tokenize_fragment_file(p, tok[1], device_parse=True)
        assert _line_of(str(dev.value)) == want and "Invalid fragment file detected" in str(dev.value)
    from gtars_b200 import ffi
    gz = bgzf_fast(bad, block=4096)
    for call in (lambda: ix.tokenize_fragments_file(bad, names, unk),
                 lambda: ix.tokenize_fragments_file(gz, names, unk, gz_member_offsets=ffi.gzip_members(gz))):
        with pytest.raises(ffi.GtarsGpuError) as e:
            call()
        assert e.value.code == 1 and _line_of(str(e.value)) == want
        b, o, i = ix.tokenize_fragments_file(good, names, unk)        # the index is usable after the failure
        tb, to, ti = ix.tokenize_fragments_text(good, names, unk)
        assert b == tb and np.array_equal(o, to) and np.array_equal(i, ti)


def _dense_first_appearance(b):
    uniq, first = np.unique(b, return_index=True)
    order = np.argsort(first, kind="stable")
    dense = np.empty(int(b.max()) + 1, dtype=np.uint32)
    dense[uniq[order]] = np.arange(order.size, dtype=np.uint32)
    return uniq[order], dense


def test_text_past_4_gib(api, universe_index, tmp_path):
    """One plain text of > 4 GiB (1.1e8 fragments) in the default 2 GiB windows == gtgpu_tokenize_fragments on the arrays
    with dense first-appearance barcode ids, through the ffi and through the Python API; the < 4 GiB text form refuses it."""
    from gtars_b200 import ffi, synth
    ix, u = universe_index
    unk = int(u["unk_id"])
    n, chunk, L = 110_000_000, 10_000_000, synth.FRAGMENT_LINE
    text = np.empty(n * L, dtype=np.uint8)
    cols = [np.empty(n, dtype=np.uint32) for _ in range(4)]
    for a in range(0, n, chunk):
        c, s, e, b = synth.make_fragment_arrays(min(chunk, n - a), 2000 + a // chunk, 10**6)
        text[a * L:(a + len(s)) * L] = synth.fragment_text(c, s, e, b)
        for dst, src in zip(cols, (c, s, e, b)):
            dst[a:a + len(s)] = src
    assert text.nbytes > 4 << 30
    order, dense = _dense_first_appearance(cols[3])
    want_off, want_ids = ix.tokenize_fragments(cols[0], cols[1], cols[2], dense[cols[3]], order.size, unk)
    names, off, ids = ix.tokenize_fragments_file(text, synth.CHROM_NAMES, unk)
    assert names == ["BC%07d" % x for x in order]
    assert np.array_equal(off, want_off) and np.array_equal(ids, want_ids)
    blob, noff = ffi._names_blob(synth.CHROM_NAMES)                  # the text form, without copying the text into bytes
    nb, h = C.c_uint32(0), [C.c_void_p() for _ in range(3)]
    st = ffi.lib().gtgpu_tokenize_fragments_text(ix._h, ffi._p(text), text.nbytes, len(synth.CHROM_NAMES), blob, ffi._p(noff), unk,
                                                 C.byref(nb), *(C.byref(x) for x in h))
    assert st == 6 and "at most 4 GiB" in ffi.lib().gtgpu_last_error().decode()
    # the same file through the host layer: a universe BED of the index's regions, so every barcode has as many ids
    cols = None
    uc, us, ue = (u[k].numpy() for k in ("chr", "start", "end"))
    uni, frag = str(tmp_path / "universe.bed"), str(tmp_path / "big.tsv")
    with open(uni, "w") as f:
        f.write("".join(f"{synth.CHROM_NAMES[x]}\t{y}\t{z}\n" for x, y, z in zip(uc, us, ue)))
    text.tofile(frag)
    del text
    got = api.tokenize_fragment_file(frag, api.Tokenizer(uni), device_parse=True)
    assert list(got) == names
    assert np.array_equal(np.fromiter((len(v) for v in got.values()), dtype=np.uint64, count=len(got)), np.diff(want_off))


def test_bgzf_at_scale(universe_index):
    """3e7 fragments as BGZF through gtgpu_tokenize_fragments_file_gz == the text form == the array entry point."""
    from gtars_b200 import ffi, synth
    ix, u = universe_index
    unk = int(u["unk_id"])
    c, s, e, b = synth.make_fragment_arrays(30_000_000, 78, 400_000)
    text = synth.fragment_text(c, s, e, b)
    gz = bgzf_fast(text)
    g = ix.tokenize_fragments_file(gz, synth.CHROM_NAMES, unk, gz_member_offsets=ffi.gzip_members(gz))
    t = ix.tokenize_fragments_file(text, synth.CHROM_NAMES, unk)
    assert g[0] == t[0] and np.array_equal(g[1], t[1]) and np.array_equal(g[2], t[2])
    order, dense = _dense_first_appearance(b)
    want_off, want_ids = ix.tokenize_fragments(c, s, e, dense[b], order.size, unk)
    assert t[0] == ["BC%07d" % x for x in order]
    assert np.array_equal(t[1], want_off) and np.array_equal(t[2], want_ids)


def test_multi_device_context_equals_single(universe_index):
    from gtars_b200 import ffi, synth
    if ffi.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    ix1, u = universe_index
    unk = int(u["unk_id"])
    offs = u["chrom_offsets"].numpy().astype(np.uint64)
    s, e, v = (u[k].numpy().view(np.uint32) for k in ("g_start", "g_end", "g_val"))
    ctx = ffi.Context(devices=[0, 1])
    ixm = ffi.Index(ctx, ffi.KIND_BITS, offs, s, e, v)
    text = synth.fragment_text(*synth.make_fragment_arrays(2_000_000, 6, 5000))
    gz = bgzf_fast(text)
    for kw in ({}, {"gz_member_offsets": ffi.gzip_members(gz)}):
        src = gz if kw else text
        a, b = ixm.tokenize_fragments_file(src, synth.CHROM_NAMES, unk, **kw), ix1.tokenize_fragments_file(src, synth.CHROM_NAMES, unk, **kw)
        assert a[0] == b[0] and np.array_equal(a[1], b[1]) and np.array_equal(a[2], b[2])
    ixm.close()
    ctx.close()
