"""count_fragments_by_barcode from a fragment file's text or gzip bytes (gtgpu_count_fragments_file / _gz, and
api.count_fragments_by_barcode with device_parse=True), parsed, tokenized and counted on the device, against a Counter over the
oracle's tokenize_fragment_file per barcode, the host path (device_parse=False) and the ids of gtgpu_tokenize_fragments_file."""
import ctypes as C
import os
from collections import Counter

import numpy as np
import pytest

from tests.test_gpu_fragment_file_text import UNIVERSE, _dense_first_appearance, _line_of, bgzf_fast
from tests.test_gpu_score_text import _pad_to, _window_text, cases, random_lines, variants

pytestmark = pytest.mark.gpu

NAMES = ["chr1", "chr2", "chrX"]
# nested and overlapping peaks: most fragments have several hits, more than the find's first capacity guess
NESTED = ("chr1\t0\t100000\nchr1\t10\t90000\nchr1\t20\t80000\nchr1\t100\t200\nchr1\t150\t400\nchr1\t1000\t1100\n"
          "chr1\t5000\t9000\nchr2\t50\t80\nchr2\t0\t7000\nchrX\t10\t4000\nchrX\t20\t30\n")


@pytest.fixture(scope="module")
def api():
    from gtars_b200 import api as a
    a.device(0)
    return a


def _tokenizers(api, d, name, text, ailist=False):
    uni = str(d / f"{name}.bed")
    with open(uni, "w") as f:
        f.write(text)
    if not ailist:
        return uni, api.Tokenizer(uni)
    toml = str(d / f"{name}.toml")
    with open(toml, "w") as f:
        f.write(f'universe = "{name}.bed"\ntokenizer_type = "ailist"\n')
    return uni, api.Tokenizer.from_config(toml)


@pytest.fixture(scope="module")
def tok(api, tmp_path_factory):
    return _tokenizers(api, tmp_path_factory.mktemp("uni"), "universe", UNIVERSE)


@pytest.fixture(scope="module")
def small_index():
    """An ffi index over UNIVERSE (val = line index, unk = 9), chromosome names in the order the text forms take them."""
    from gtars_b200 import ffi
    rows = [l.split("\t") for l in UNIVERSE.splitlines()]
    offs = np.array([0, 5, 7, 9], dtype=np.uint64)
    s, e = (np.array([int(r[k]) for r in rows], dtype=np.uint32) for k in (1, 2))
    ctx = ffi.Context(0)
    ix = ffi.Index(ctx, ffi.KIND_BITS, offs, s, e, np.arange(len(rows), dtype=np.uint32))
    yield ix, NAMES, len(rows)
    ix.close()
    ctx.close()


def oracle_counts(uni, path, ailist=False):
    from oracle import oracle as orc
    t = orc.Tokenizer(uni, orc.AILIST if ailist else orc.BITS)
    return {bc: dict(Counter(ids)) for bc, ids in t.tokenize_fragment_file(path).items()}


def same_counts(api, tok, path, ailist=False):
    """device_parse=True == device_parse=False (equal dicts, equal barcode order) == the oracle; barcodes in the order
    tokenize_fragment_file gives them, every barcode's token ids ascending."""
    uni, t = tok
    dev = api.count_fragments_by_barcode(path, t, device_parse=True)
    host = api.count_fragments_by_barcode(path, t)
    assert dev == host and list(dev) == list(host), path
    assert list(dev) == list(api.tokenize_fragment_file(path, t, device_parse=True)), path
    assert all(list(v) == sorted(v) and all(c > 0 for c in v.values()) for v in dev.values()), path
    assert dev == oracle_counts(uni, path, ailist), path
    return dev


def counts_from_ids(off, ids):
    """The CSR gtgpu_count_fragments_file returns, computed from gtgpu_tokenize_fragments_file's (offsets, ids)."""
    off = off.astype(np.int64)
    bc = np.repeat(np.arange(len(off) - 1, dtype=np.uint64), np.diff(off))
    m = np.uint64(int(ids.max()) + 1 if len(ids) else 1)
    keys, cnt = np.unique(bc * m + ids.astype(np.uint64), return_counts=True)
    return (np.searchsorted(keys // m, np.arange(len(off), dtype=np.uint64)).astype(np.uint64), (keys % m).astype(np.uint32),
            cnt.astype(np.uint32))


def count_file_form(ix, names, unk, text):
    """gtgpu_count_fragments_file on the text and _gz on its BGZF form, both equal to the counts of the tokenize form's ids."""
    from gtars_b200 import ffi
    got = ix.count_fragments_file(text, names, unk)
    gz = bgzf_fast(bytes(text), block=min(65_280, max(64, -(-len(text) // 20))))
    got_gz = ix.count_fragments_file(gz, names, unk, gz_member_offsets=ffi.gzip_members(gz))
    assert got_gz[0] == got[0] and all(np.array_equal(a, b) for a, b in zip(got_gz[1:], got[1:]))
    b, o, i = ix.tokenize_fragments_file(text, names, unk)
    assert got[0] == b
    want = counts_from_ids(o, i)
    assert all(np.array_equal(a, w) for a, w in zip(got[1:], want))
    assert len(got[1]) == len(got[0]) + 1 and got[1][-1] == len(got[2]) == len(got[3])
    return got


def test_kat_d3(api, golden, fixture_dir, tmp_path):
    """D3 (the reference's fragment fixture) as plain text, BGZF and single-member gzip: the Counter of each barcode's ids."""
    import gzip
    d3 = golden[1]["D_derived"]["D3"]
    uni = os.path.join(fixture_dir, d3["universe"])
    t = api.Tokenizer(uni)
    src = os.path.join(fixture_dir, d3["fragments"])
    with open(src, "rb") as f:
        raw = f.read()
    text = gzip.decompress(raw) if src.endswith(".gz") else raw
    want = {"AAACGCAAGCAAAGGGATGCCA": {0: 2, 1: 1, 3: 2, 4: 1}, "AAACGCAAGCAACTGCGTCTTT": {0: 1, 2: 1}}
    assert want == {bc: dict(Counter(ids)) for bc, ids in d3["expect"].items()}
    for p in variants(tmp_path, "d3", text):
        got = same_counts(api, (uni, t), p)
        assert got == want and list(got) == list(want), p


@pytest.mark.parametrize("case", sorted(cases()))
def test_edge_cases(api, tok, small_index, tmp_path, case):
    """comments, whitespace and CRLF, extra columns, unknown chromosomes, no trailing newline, an empty file, '#' lines only"""
    ix, names, unk = small_index
    text = cases()[case]
    b, o, t, c = count_file_form(ix, names, unk, text)
    for p in variants(tmp_path, case, text):
        got = same_counts(api, tok, p)
        if case == "unknown_chroms":
            assert got["GHOST"] == {unk: 2} and "GHOST" in b               # seen only on unknown chromosomes: {unk: n}
        if case in ("empty", "comments_only"):
            assert got == {} and b == [] and list(o) == [0] and len(t) == len(c) == 0


def test_no_hit_fragments_count_under_unk(api, tok, small_index, tmp_path):
    """fragments with no hit (gaps, unknown and known chromosomes) each count once under unk, next to their barcode's hits"""
    ix, names, unk = small_index
    text = ("chr1\t10\t20\tA\t1\nchr1\t2000\t3000\tA\t1\nchr9\t1\t2\tA\t1\nchr1\t100\t120\tA\t1\nchr2\t0\t10\tB\t1\n"
            "chrUn\t5\t6\tC\t1\nchrUn\t5\t6\tC\t1\nchrX\t4294967290\t4294967295\tB\t1\n").encode()
    b, o, t, c = count_file_form(ix, names, unk, text)
    assert b == ["A", "B", "C"]
    for p in variants(tmp_path, "nohit", text):
        assert same_counts(api, tok, p) == {"A": {1: 1, unk: 3}, "B": {8: 1, unk: 1}, "C": {unk: 2}}


def test_windows_give_the_single_window_result(api, tok, small_index, tmp_path, monkeypatch):
    """Windows of 1 byte to 64 KiB: barcodes whose fragments lie in many windows, and barcodes that first appear late."""
    ix, names, unk = small_index
    rng = np.random.default_rng(51)
    body = "\n".join(_window_text(rng)) + "\n"
    head = "chr1\t120\t130\tFIRST\t1"
    texts = {"nl": _pad_to(head, "\n", False) + body + head + "\n", "crlf": _pad_to(head, "\r", True) + body,
             "comment": head + "\n" + "#" + "c" * 2000 + "\n" + body}
    texts = {k: v.encode() for k, v in texts.items()}
    paths = {k: variants(tmp_path, k, v)[:2] for k, v in texts.items()}
    monkeypatch.delenv("GTGPU_INGEST_WINDOW", raising=False)
    want = {k: count_file_form(ix, names, unk, v) for k, v in texts.items()}
    want_api = {k: [same_counts(api, tok, p) for p in ps] for k, ps in paths.items()}
    assert want_api["nl"][0]["FIRST"][1] >= 2                         # FIRST in the first and the last window
    for w in ("1", "1024", "4096", "65536"):
        monkeypatch.setenv("GTGPU_INGEST_WINDOW", w)
        for k, v in texts.items():
            got = count_file_form(ix, names, unk, v)
            assert got[0] == want[k][0] and all(np.array_equal(x, y) for x, y in zip(got[1:], want[k][1:])), (w, k)
            for p, d in zip(paths[k], want_api[k]):
                got_api = api.count_fragments_by_barcode(p, tok[1], device_parse=True)
                assert got_api == d and list(got_api) == list(d), (w, k, p)


def test_nested_universe_bits_and_ailist(api, tmp_path):
    """Multi-hit fragments (several per fragment: the find re-runs with an exact buffer) give equal counts with Bits and AIList."""
    rng = np.random.default_rng(52)
    text = ("\n".join(random_lines(rng, 6000, names=("chr1", "chr1", "chr2", "chr9"), n_bc=700)) + "\n").encode()
    bits = _tokenizers(api, tmp_path, "nested", NESTED)
    ail = _tokenizers(api, tmp_path, "nested", NESTED, ailist=True)
    for p in variants(tmp_path, "nested_frags", text):
        a = same_counts(api, bits, p)
        b = same_counts(api, ail, p, ailist=True)
        assert a == b and list(a) == list(b), p
        assert sum(sum(v.values()) for v in a.values()) > 6000 * 5 // 4 + 1024   # more tokens than the first capacity
        assert len(a) > 512                                              # barcode ids of 10 bits: two digit passes


def test_duplicate_universe_lines(api, tmp_path):
    """A region listed twice is one token id that a fragment over it hits twice."""
    uni_text = "chr1\t100\t200\nchr1\t100\t200\nchr1\t150\t400\nchr2\t50\t80\nchr1\t150\t400\nchrX\t10\t4000\n"
    t = _tokenizers(api, tmp_path, "dups", uni_text)
    rng = np.random.default_rng(53)
    text = ("\n".join(random_lines(rng, 400, n_bc=30)) + "\nchr1\t120\t130\tDUP\t1\n").encode()
    for p in variants(tmp_path, "dups", text):
        assert "DUP" in same_counts(api, t, p)


@pytest.mark.parametrize("n_regions", [8, 256, 512])
def test_unk_needs_a_bit_max_val_does_not(api, tmp_path, n_regions):
    """A universe of exactly 2^k regions: unk_id = 2^k is one bit wider than every region id (at 256 and 512 that bit is also a
    radix digit of its own), so the token sort runs on max(max_val, unk_id)'s bits."""
    uni_text = "".join(f"chr1\t{i * 100}\t{i * 100 + 50}\n" for i in range(n_regions))
    t = _tokenizers(api, tmp_path, f"u{n_regions}", uni_text)
    assert t[1].unk_token_id == n_regions
    rng = np.random.default_rng(n_regions)
    lines = []
    for k in range(3000):
        c = ["chr1", "chr1", "chr1", "chr2"][k % 4]
        s = int(rng.integers(0, n_regions * 100 + 300))
        lines.append(f"{c}\t{s}\t{s + int(rng.integers(1, 40))}\tB{int(rng.integers(0, 25))}\t1")
    for p in variants(tmp_path, f"u{n_regions}_frags", ("\n".join(lines) + "\n").encode()):
        got = same_counts(api, t, p)
        assert all(n_regions in v for v in got.values())                  # every barcode has no-hit fragments
        assert any(n_regions - 1 in v for v in got.values())


def test_malformed_line(api, tok, small_index, tmp_path, monkeypatch):
    """A short line in a late window: the 0-based line index of the host path, no output, and the next call succeeds."""
    from gtars_b200 import ffi
    ix, names, unk = small_index
    rng = np.random.default_rng(54)
    lines = _window_text(rng)
    good = ("\n".join(lines) + "\n").encode()
    lines.insert(len(lines) - 40, "chr2\t1\t2\tLATE")
    bad = ("\n".join(lines) + "\n").encode()
    ps = variants(tmp_path, "late", bad)
    with pytest.raises(api.GtarsError) as host:
        api.count_fragments_by_barcode(ps[0], tok[1])
    want = _line_of(str(host.value))
    assert want == len(lines) - 41
    monkeypatch.setenv("GTGPU_INGEST_WINDOW", "1024")
    for p in ps:
        with pytest.raises(api.GtarsError) as dev:
            api.count_fragments_by_barcode(p, tok[1], device_parse=True)
        assert _line_of(str(dev.value)) == want and "Invalid fragment file detected" in str(dev.value)
    blob, noff = ffi._names_blob(names)
    gz = bgzf_fast(bad, block=4096)
    mo = ffi.gzip_members(gz)
    calls = (lambda outs: ffi.lib().gtgpu_count_fragments_file(ix._h, bad, len(bad), len(names), blob, ffi._p(noff), unk, *outs),
             lambda outs: ffi.lib().gtgpu_count_fragments_file_gz(ix._h, len(mo) - 1, gz, ffi._p(mo), len(names), blob, ffi._p(noff),
                                                                  unk, *outs))
    for call in calls:
        nb, hs = C.c_uint32(0), [C.c_void_p() for _ in range(5)]
        st = call((C.byref(nb),) + tuple(C.byref(h) for h in hs))
        msg = ffi.lib().gtgpu_last_error().decode()
        assert st == 1 and _line_of(msg) == want and "Invalid fragment file detected" in msg
        assert nb.value == 0 and all(h.value is None for h in hs)       # no output
        count_file_form(ix, names, unk, good)                             # the index is usable after the failure
    monkeypatch.delenv("GTGPU_INGEST_WINDOW")
    assert same_counts(api, tok, variants(tmp_path, "good", good)[0])


# ---- a synth universe of 2e5 regions -----------------------------------------------------------------------------------------
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


@pytest.mark.parametrize("n,n_barcodes", [(1_000_000, 1000), (10_000_000, 400_000)])
def test_synth_at_scale(universe_index, n, n_barcodes):
    """1e6 fragments over 1 000 barcodes (two radix digit passes by barcode) and 1e7 over 4e5 (three), plain and BGZF: the counts
    of gtgpu_tokenize_fragments_file's ids, barcodes in the order of the arrays' first appearance."""
    from gtars_b200 import synth
    ix, u = universe_index
    unk = int(u["unk_id"])
    c, s, e, b = synth.make_fragment_arrays(n, 91 + n_barcodes, n_barcodes)
    text = synth.fragment_text(c, s, e, b)
    names, off, tokens, counts = count_file_form(ix, synth.CHROM_NAMES, unk, text)
    order, _ = _dense_first_appearance(b)
    assert names == ["BC%07d" % x for x in order]
    bits = (len(names) - 1).bit_length()                              # radix digits of <= 9 bits
    assert 10 <= bits <= 18 if n_barcodes == 1000 else bits >= 19
    assert int(counts.sum(dtype=np.uint64)) >= n and (tokens == unk).any() and (tokens < unk).any()


def test_synth_slice_through_the_api(api, tmp_path):
    """2e5 fragments against a universe file of 2e5 synth regions, through the host layer, against the oracle."""
    from gtars_b200 import synth
    u = synth.make_universe(200_000)
    uc, us, ue = (u[k].numpy() for k in ("chr", "start", "end"))
    uni = str(tmp_path / "universe.bed")
    with open(uni, "w") as f:
        f.write("".join(f"{synth.CHROM_NAMES[x]}\t{y}\t{z}\n" for x, y, z in zip(uc, us, ue)))
    path = str(tmp_path / "slice.tsv")
    synth.fragment_text(*synth.make_fragment_arrays(200_000, 92, 5000)).tofile(path)
    got = same_counts(api, (uni, api.Tokenizer(uni)), path)
    assert len(got) > 4000


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
    text = synth.fragment_text(*synth.make_fragment_arrays(2_000_000, 93, 5000))
    a, b = ixm.count_fragments_file(text, synth.CHROM_NAMES, unk), ix1.count_fragments_file(text, synth.CHROM_NAMES, unk)
    assert a[0] == b[0] and all(np.array_equal(x, y) for x, y in zip(a[1:], b[1:]))
    ixm.close()
    ctx.close()
