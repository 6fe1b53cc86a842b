"""The argument rules of the 16 device text entry points (eight operations, each on plain text and on gzip members): every
malformed input is rejected with GTGPU_ERR_INVALID under the entry point's own name, and the context serves a valid call
afterwards."""
import ctypes as C
import gzip

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ERR_INVALID = 1
NAMES = ["chr1", "chr2"]
BED = b"chr1\t100\t200\nchr2\t50\t80\nchr1\t10\t20\n"
FRAG = b"chr1\t100\t200\tAAA\t1\nchr2\t50\t80\tCCC\t2\nchr1\t150\t160\tAAA\t1\n"


class Plain:
    """text (None: a null pointer), n_bytes; file_offsets for the entry points that take several files"""

    def __init__(self, body, n_files=2, text=True, fo=None):
        self.text = body * n_files if text else None
        self.n_bytes = len(body) * n_files
        self.fo = np.array(fo if fo is not None else [len(body) * f for f in range(n_files + 1)], dtype=np.uint64)
        self.n_files = len(self.fo) - 1


class Gz:
    """gz (None: a null pointer), member_offsets (n_members + 1), file_members for the entry points that take several files"""

    def __init__(self, body, n_members=2, gz=True, mo=None, fm=None):
        members = [gzip.compress(body, mtime=0) for _ in range(n_members)]
        self.gz = b"".join(members) if gz else None
        self.mo = np.array(mo if mo is not None else np.cumsum([0] + [len(m) for m in members]), dtype=np.uint64)
        self.n_members = len(self.mo) - 1
        self.fm = np.array(fm if fm is not None else range(n_members + 1), dtype=np.uint64)
        self.n_files = len(self.fm) - 1


class Outs:
    """output handles of one call, freed after it"""

    def __init__(self):
        self.bufs, self.igds = [], []

    def buf(self):
        self.bufs.append(C.c_void_p())
        return C.byref(self.bufs[-1])

    def igd(self):
        self.igds.append(C.c_void_p())
        return C.byref(self.igds[-1])

    def free(self, L):
        for h in self.bufs:
            if h.value:
                L.gtgpu_buf_free(h)
        for h in self.igds:
            if h.value:
                L.gtgpu_igd_free(h)


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def _call(fx, name, t):
    """gtgpu_<name> on input t with valid other arguments; returns the status"""
    from gtars_b200 import ffi
    L = ffi.lib()
    blob, no = ffi._names_blob(NAMES)
    nn, ix, unk, o = len(NAMES), fx["index"], 7, Outs()
    u32 = C.c_uint32()
    tok = np.zeros(max(t.n_files, 0) + 1, dtype=np.uint64)
    row = np.zeros(8, dtype=np.uint32)
    mat = np.zeros((max(t.n_files, 1), 2), dtype=np.uint64)
    reg = np.zeros(max(t.n_files, 1), dtype=np.uint64)
    calls = {
        "tokenize_bed": lambda: L.gtgpu_tokenize_bed(ix, t.text, t.n_bytes, nn, blob, _p(no), unk, o.buf()),
        "tokenize_bed_gz": lambda: L.gtgpu_tokenize_bed_gz(ix, t.n_members, t.gz, _p(t.mo), nn, blob, _p(no), unk, o.buf()),
        "tokenize_bed_files": lambda: L.gtgpu_tokenize_bed_files(ix, t.n_files, t.text, _p(t.fo), nn, blob, _p(no), unk, _p(tok),
                                                                 o.buf()),
        "tokenize_bed_files_gz": lambda: L.gtgpu_tokenize_bed_files_gz(ix, t.n_files, _p(t.fm), t.n_members, t.gz, _p(t.mo), nn, blob,
                                                                       _p(no), unk, _p(tok), o.buf()),
        "tokenize_fragments_text": lambda: L.gtgpu_tokenize_fragments_text(ix, t.text, t.n_bytes, nn, blob, _p(no), unk, C.byref(u32),
                                                                           o.buf(), o.buf(), o.buf()),
        "tokenize_fragments_gz": lambda: L.gtgpu_tokenize_fragments_gz(ix, t.n_members, t.gz, _p(t.mo), nn, blob, _p(no), unk,
                                                                       C.byref(u32), o.buf(), o.buf(), o.buf(), o.buf()),
        "tokenize_fragments_file": lambda: L.gtgpu_tokenize_fragments_file(ix, t.text, t.n_bytes, nn, blob, _p(no), unk, C.byref(u32),
                                                                           o.buf(), o.buf(), o.buf(), o.buf()),
        "tokenize_fragments_file_gz": lambda: L.gtgpu_tokenize_fragments_file_gz(ix, t.n_members, t.gz, _p(t.mo), nn, blob, _p(no), unk,
                                                                                 C.byref(u32), o.buf(), o.buf(), o.buf(), o.buf()),
        "score_matrix_text": lambda: L.gtgpu_score_matrix_text(ix, t.text, t.n_bytes, nn, blob, _p(no), ffi.SCORE_CHIP, len(row),
                                                               _p(row)),
        "score_matrix_gz": lambda: L.gtgpu_score_matrix_gz(ix, t.n_members, t.gz, _p(t.mo), nn, blob, _p(no), ffi.SCORE_CHIP, len(row),
                                                           _p(row)),
        "score_barcodes_text": lambda: L.gtgpu_score_barcodes_text(ix, t.text, t.n_bytes, nn, blob, _p(no), C.byref(u32), o.buf(),
                                                                   o.buf(), o.buf(), o.buf(), o.buf()),
        "score_barcodes_gz": lambda: L.gtgpu_score_barcodes_gz(ix, t.n_members, t.gz, _p(t.mo), nn, blob, _p(no), C.byref(u32), o.buf(),
                                                               o.buf(), o.buf(), o.buf(), o.buf()),
        "igd_build_bed": lambda: L.gtgpu_igd_build_bed(fx["ctx"], t.n_files, t.text, _p(t.fo), C.byref(u32), o.buf(), o.buf(), o.igd()),
        "igd_build_bed_gz": lambda: L.gtgpu_igd_build_bed_gz(fx["ctx"], t.n_files, _p(t.fm), t.n_members, t.gz, _p(t.mo), C.byref(u32),
                                                             o.buf(), o.buf(), o.igd()),
        "igd_count_bed": lambda: L.gtgpu_igd_count_bed(fx["igd"], 0, t.n_files, t.text, _p(t.fo), nn, blob, _p(no), 1, _p(mat),
                                                       _p(reg)),
        "igd_count_bed_gz": lambda: L.gtgpu_igd_count_bed_gz(fx["igd"], 0, t.n_files, _p(t.fm), t.n_members, t.gz, _p(t.mo), nn, blob,
                                                             _p(no), 1, _p(mat), _p(reg)),
    }
    try:
        return calls[name]()
    finally:
        o.free(L)


# entry point -> (format of its text, takes several files)
ENTRY = {
    "tokenize_bed": (BED, False), "tokenize_bed_files": (BED, True), "tokenize_fragments_text": (FRAG, False),
    "tokenize_fragments_file": (FRAG, False), "score_matrix_text": (FRAG, False), "score_barcodes_text": (FRAG, False),
    "igd_build_bed": (BED, True), "igd_count_bed": (BED, True),
    "tokenize_bed_gz": (BED, False), "tokenize_bed_files_gz": (BED, True), "tokenize_fragments_gz": (FRAG, False),
    "tokenize_fragments_file_gz": (FRAG, False), "score_matrix_gz": (FRAG, False), "score_barcodes_gz": (FRAG, False),
    "igd_build_bed_gz": (BED, True), "igd_count_bed_gz": (BED, True),
}


def _is_gz(name):
    return name.endswith("_gz")


# case -> (applies to (gz?, several files?), input builder(body), expected message part: None = the entry point's name)
CASES = {
    "null_text": (lambda gz, files: not gz, lambda b, files: Plain(b, text=False) if files else Plain(b, 1, text=False), None),
    "null_gz": (lambda gz, files: gz, lambda b, files: Gz(b, gz=False), None),
    "file_offsets_not_from_0": (lambda gz, files: not gz and files, lambda b, files: Plain(b, fo=[1, len(b), 2 * len(b)]), None),
    "file_offsets_not_monotone": (lambda gz, files: not gz and files, lambda b, files: Plain(b, fo=[0, 2 * len(b), len(b)]), None),
    "member_offsets_not_monotone": (lambda gz, files: gz, lambda b, files: Gz(b, mo=[0, Gz(b).mo[2], Gz(b).mo[1]]), None),
    "file_members_not_ending_at_n_members": (lambda gz, files: gz and files, lambda b, files: Gz(b, fm=[0, 1, 1]), None),
    "file_members_not_from_0": (lambda gz, files: gz and files, lambda b, files: Gz(b, fm=[1, 1, 2]), None),
    "file_members_not_monotone": (lambda gz, files: gz and files, lambda b, files: Gz(b, fm=[0, 2, 1, 2]), None),
    "short_member": (lambda gz, files: gz, lambda b, files: Gz(b, mo=[0, Gz(b).mo[1], Gz(b).mo[1] + 17]), "member 1"),
}

PAIRS = [(e, c) for e, (body, files) in ENTRY.items() for c, (applies, _, _) in CASES.items() if applies(_is_gz(e), files)]


@pytest.fixture(scope="module")
def fx():
    from gtars_b200 import ffi
    ctx = ffi.Context(0)
    offs = np.array([0, 2, 3], dtype=np.uint64)
    ix = ffi.Index(ctx, ffi.KIND_BITS, offs, np.array([90, 180, 40], np.uint32), np.array([150, 300, 60], np.uint32))
    igd, names = ffi.Igd.from_bed_text(ctx, BED * 2, [0, len(BED), 2 * len(BED)])
    assert names == NAMES
    yield {"ctx": ctx._h, "index": ix._h, "igd": igd._h}
    igd.close()
    ix.close()
    ctx.close()


def _valid(name):
    body, files = ENTRY[name]
    return Gz(body) if _is_gz(name) else Plain(body, 2 if files else 1)


@pytest.mark.parametrize("name", list(ENTRY))
def test_valid_input_is_accepted(fx, name):
    from gtars_b200 import ffi
    assert _call(fx, name, _valid(name)) == 0, ffi.lib().gtgpu_last_error().decode()


@pytest.mark.parametrize("name,case", PAIRS)
def test_malformed_input_is_rejected(fx, name, case):
    """the malformed input fails with GTGPU_ERR_INVALID under the entry point's name (or gunzip's member text); a valid call
    on the same context then succeeds"""
    from gtars_b200 import ffi
    L = ffi.lib()
    body, files = ENTRY[name]
    _, make, want = CASES[case]
    assert _call(fx, name, make(body, files)) == ERR_INVALID
    msg = L.gtgpu_last_error().decode()
    if want is None:
        assert msg.startswith(name + ": "), msg
    else:
        assert want in msg, msg
    assert _call(fx, name, _valid(name)) == 0, L.gtgpu_last_error().decode()

