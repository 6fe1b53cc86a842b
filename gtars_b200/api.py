"""Python face of the C++ host layer (libgtars_host.so): the reference's public names for the interval-overlap path.

    gtars.tokenizers.Tokenizer          -> Tokenizer          (gtars-python/src/tokenizers/py_tokenizers/mod.rs:14-300)
    gtars.models.Region / RegionSet     -> Region, RegionSet  (gtars-python/src/models/region_set.rs:445-481)
    gtars_overlaprs MultiChromOverlapper / IndexedRegionSet -> MultiChromOverlapper
    gtars.tokenizers.tokenize_fragment_file                 -> tokenize_fragment_file
    gtars-tokenizers count_fragments_by_barcode             -> count_fragments_by_barcode
    gtars.lola RegionDB / run_lola (contingency counts)     -> Igd, lola_contingency, lola_contingency_from_bed_files

Every batch method is one call into the C++ layer, which marshals to the C ABI of include/gtars_gpu.h; nothing here
(or below) computes an overlap on the CPU, and construction fails without a CUDA device.
"""
from __future__ import annotations

import ctypes as C
import os
from dataclasses import dataclass

import numpy as np

_PKG = os.path.dirname(os.path.abspath(__file__))
HOST_LIB_PATH = os.path.join(_PKG, "libgtars_host.so")
BITS, AILIST = 0, 1
_lib = None


class GtarsError(RuntimeError):
    pass


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(HOST_LIB_PATH):
            raise ImportError(f"{HOST_LIB_PATH} is missing: run `make -C gtars_b200/csrc all`")
        C.CDLL(os.path.join(_PKG, "libgtars_gpu.so"), mode=C.RTLD_GLOBAL)
        L = C.CDLL(HOST_LIB_PATH)
        vp, u64, u32, i32, i64, cp = C.c_void_p, C.c_uint64, C.c_uint32, C.c_int32, C.c_int64, C.c_char_p
        sig = {
            "gth_last_error": (cp, []), "gth_device_new": (vp, [C.c_int]), "gth_device_free": (None, [vp]),
            "gth_regionset_from_file": (vp, [cp]), "gth_regionset_new": (vp, [u64, vp, vp, vp]),
            "gth_regionset_free": (None, [vp]), "gth_regionset_len": (u64, [vp]), "gth_regionset_chr": (cp, [vp, u64]),
            "gth_regionset_start": (u32, [vp, u64]), "gth_regionset_end": (u32, [vp, u64]),
            "gth_lists_free": (None, [vp]), "gth_lists_n": (u64, [vp]), "gth_lists_len": (u64, [vp, u64]),
            "gth_lists_data": (vp, [vp, u64]), "gth_lists_name": (cp, [vp, u64]),
            "gth_mco_new": (vp, [vp, vp, C.c_int]), "gth_mco_free": (None, [vp]), "gth_mco_count": (C.c_int, [vp, vp, i32, vp]),
            "gth_mco_any": (C.c_int, [vp, vp, i32, vp]), "gth_mco_find": (vp, [vp, vp, i32]),
            "gth_mco_subset_by": (vp, [vp, vp, i32]),
            "gth_irs_new": (vp, [vp, vp, C.c_int]), "gth_irs_free": (None, [vp]), "gth_irs_find": (vp, [vp, vp, i32]),
            "gth_irs_subset_by_overlaps": (vp, [vp, vp, i32]), "gth_irs_count": (C.c_int, [vp, vp, i32, vp]),
            "gth_irs_any": (C.c_int, [vp, vp, i32, vp]),
            "gth_consensus_new": (vp, [vp, cp]), "gth_consensus_free": (None, [vp]), "gth_consensus_len": (u64, [vp]),
            "gth_region_scoring": (C.c_int, [vp, u64, vp, C.c_int, vp]), "gth_barcode_scoring": (vp, [vp, cp]),
            "gth_region_scoring_device": (C.c_int, [vp, u64, vp, C.c_int, vp]), "gth_barcode_scoring_device": (vp, [vp, cp]),
            "gth_tokenizer_new": (vp, [vp, cp, C.c_int]), "gth_tokenizer_free": (None, [vp]),
            "gth_tokenizer_vocab_size": (u64, [vp]), "gth_tokenizer_token_to_id": (i64, [vp, cp]),
            "gth_tokenizer_id_to_token": (cp, [vp, u32]), "gth_tokenizer_special": (cp, [vp, C.c_int]),
            "gth_tokenizer_kind": (C.c_int, [vp]), "gth_tokenizer_encode_batch": (vp, [vp, u64, vp]),
            "gth_tokenizer_fragments": (vp, [vp, cp]), "gth_tokenizer_fragments_device": (vp, [vp, cp]), "gth_tokenizer_encode_bed_file": (vp, [vp, cp]),
            "gth_tokenizer_encode_bed_files": (vp, [vp, u64, vp]),
            "gth_tokenizer_count_fragments": (vp, [vp, cp]), "gth_tokenizer_count_fragments_device": (vp, [vp, cp]),
            "gth_parse_bed_file": (vp, [vp, cp, u64, vp]), "gth_gtok_write": (C.c_int, [cp, u64, vp, C.c_int]),
            "gth_gtok_read": (vp, [cp]),
            "gth_igd_single": (vp, [vp, vp]), "gth_igd_find_pairs": (vp, [vp, vp, i32]),
            "gth_igd_count_per_query": (vp, [vp, vp, i32]),
            "gth_igd_save_sets": (C.c_int, [u64, vp, vp, cp]), "gth_igd_save": (C.c_int, [vp, u64, vp, cp]),
            "gth_igd_from_file": (vp, [vp, cp]),
            "gth_igd_from_bed_files": (vp, [vp, u64, vp]), "gth_igd_info": (C.c_int, [vp, vp]),
            "gth_igd_new": (vp, [vp, u64, vp]), "gth_igd_free": (None, [vp]), "gth_igd_num_files": (u64, [vp]),
            "gth_igd_count": (C.c_int, [vp, u64, vp, i32, C.c_int, vp]),
            "gth_lola_contingency": (C.c_int, [vp, u64, vp, vp, i32, vp]),
            "gth_igd_count_bed_files": (C.c_int, [vp, u64, vp, i32, C.c_int, vp, vp]),
            "gth_lola_contingency_bed_files": (C.c_int, [vp, u64, vp, cp, i32, vp]),
            "gth_mco_overlaps_bed_files": (vp, [vp, u64, vp, C.c_int, i32]), "gth_irs_find_bed_files": (vp, [vp, u64, vp, i32]),
            "gth_overlaps_free": (None, [vp]), "gth_overlaps_len": (u64, [vp, C.c_int]), "gth_overlaps_data": (vp, [vp, C.c_int]),
            "gth_mco_subset_by_bed_files": (C.c_int, [vp, u64, vp, i32, vp]),
            "gth_irs_subset_by_overlaps_bed_files": (C.c_int, [vp, u64, vp, i32, vp]),
        }
        for name, (res, args) in sig.items():
            fn = getattr(L, name)
            fn.restype, fn.argtypes = res, args
        _lib = L
    return _lib


def _fail():
    raise GtarsError(lib().gth_last_error().decode(errors="replace"))


_device = None


def device(index: int = 0):
    """The process-wide device handle (one GPU per process)."""
    global _device
    if _device is None:
        h = lib().gth_device_new(index)
        if not h:
            _fail()
        _device = h
    return _device


@dataclass(frozen=True)
class Region:
    chr: str
    start: int
    end: int


class RegionSet:
    """gtars_core::models::RegionSet.  RegionSet(path) parses a BED file and sorts it by (chr, start) like
    RegionSet::try_from (gtars-core/src/models/region_set.rs:60-185); RegionSet(list_of_regions) keeps the order."""

    def __init__(self, source):
        L = lib()
        if isinstance(source, (str, os.PathLike)):
            self._h = L.gth_regionset_from_file(os.fsencode(source))
        else:
            regs = [(r.chr, r.start, r.end) if isinstance(r, Region) else tuple(r) for r in source]
            chrs = (C.c_char_p * max(len(regs), 1))(*[r[0].encode() for r in regs])
            s = np.array([r[1] for r in regs], dtype=np.uint32)
            e = np.array([r[2] for r in regs], dtype=np.uint32)
            self._h = L.gth_regionset_new(len(regs), chrs, s.ctypes.data, e.ctypes.data)
        if not self._h:
            _fail()

    @classmethod
    def _wrap(cls, handle):
        obj = cls.__new__(cls)
        obj._h = handle
        return obj

    def __del__(self):
        if getattr(self, "_h", None):
            lib().gth_regionset_free(self._h)
            self._h = None

    def __len__(self):
        return lib().gth_regionset_len(self._h)

    def __getitem__(self, i):
        L = lib()
        if not 0 <= i < len(self):
            raise IndexError(i)
        return Region(L.gth_regionset_chr(self._h, i).decode(), L.gth_regionset_start(self._h, i), L.gth_regionset_end(self._h, i))

    def __iter__(self):
        return (self[i] for i in range(len(self)))

    # gtars-python/src/models/region_set.rs:445-481: `self` supplies the queries, `other` is indexed (AIList default)
    def count_overlaps(self, other: "RegionSet", min_overlap=None):
        return MultiChromOverlapper(other, AILIST).count_overlaps(self, min_overlap)

    def any_overlaps(self, other: "RegionSet", min_overlap=None):
        return MultiChromOverlapper(other, AILIST).any_overlaps(self, min_overlap)

    def find_overlaps(self, other: "RegionSet", min_overlap=None):
        return MultiChromOverlapper(other, AILIST).find_overlaps(self, min_overlap)


def _as_rs(x) -> RegionSet:
    return x if isinstance(x, RegionSet) else RegionSet(x)


def _take_lists(h, named=False):
    L = lib()
    if not h:
        _fail()
    try:
        out = []
        for i in range(L.gth_lists_n(h)):
            n = L.gth_lists_len(h, i)
            a = np.empty(n, dtype=np.uint32)
            if n:
                C.memmove(a.ctypes.data, L.gth_lists_data(h, i), 4 * n)
            vals = [int(x) for x in a]
            out.append((L.gth_lists_name(h, i).decode(), vals) if named else vals)
        return out
    finally:
        L.gth_lists_free(h)


def _paths_arg(paths):
    enc = [os.fsencode(p) for p in paths]
    return enc, (C.c_char_p * max(len(enc), 1))(*enc)


_OVERLAPS_COUNT, _OVERLAPS_ANY, _OVERLAPS_FIND = 0, 1, 2  # GTGPU_OVERLAPS_* of include/gtars_gpu.h


def _take_overlaps(h):
    """(file_queries, offsets, values, flags) of a gth_overlaps handle as NumPy arrays: one copy each, no per-element work."""
    L = lib()
    if not h:
        _fail()
    try:
        out = []
        for which, dtype in enumerate((np.uint64, np.uint64, np.uint32, np.uint8)):
            a = np.empty(L.gth_overlaps_len(h, which), dtype=dtype)
            if len(a):
                C.memmove(a.ctypes.data, L.gth_overlaps_data(h, which), a.nbytes)
            out.append(a)
        return out
    finally:
        L.gth_overlaps_free(h)


def _per_file(values, file_queries):
    """values split into one array view per file"""
    return np.split(values, file_queries[1:-1].astype(np.int64)) if len(file_queries) > 1 else []


def _per_file_hits(file_queries, offsets, vals):
    """per file (offsets from 0, vals): the file's queries' slice of a flat per-query find result"""
    out = []
    for f in range(len(file_queries) - 1):
        o = offsets[int(file_queries[f]):int(file_queries[f + 1]) + 1]
        out.append((o - o[0], vals[int(o[0]):int(o[-1])]))
    return out


def _subset_sets(fn, h, paths, min_overlap):
    enc, arr = _paths_arg(paths)
    out = (C.c_void_p * max(len(enc), 1))()
    if fn(h, len(enc), arr, min_overlap, out):
        _fail()
    return [RegionSet._wrap(out[f]) for f in range(len(enc))]


class MultiChromOverlapper:
    """gtars_overlaprs::MultiChromOverlapper over a RegionSet (val = index of the region in the source)."""

    def __init__(self, source, kind=AILIST):
        self._src = _as_rs(source)
        self._h = lib().gth_mco_new(device(), self._src._h, kind)
        if not self._h:
            _fail()

    def __del__(self):
        if getattr(self, "_h", None):
            lib().gth_mco_free(self._h)
            self._h = None

    @staticmethod
    def _m(min_overlap):
        return -1 if min_overlap is None else int(min_overlap)

    def count_overlaps(self, query, min_overlap=None):
        q = _as_rs(query)
        out = np.zeros(len(q), dtype=np.uint64)
        if lib().gth_mco_count(self._h, q._h, self._m(min_overlap), out.ctypes.data):
            _fail()
        return [int(x) for x in out]

    def any_overlaps(self, query, min_overlap=None):
        q = _as_rs(query)
        out = np.zeros(len(q), dtype=np.uint8)
        if lib().gth_mco_any(self._h, q._h, self._m(min_overlap), out.ctypes.data):
            _fail()
        return [bool(x) for x in out]

    def find_overlaps(self, query, min_overlap=None):
        """IndexedRegionSet::find_overlaps: per query, indices into the source (reference iteration order)."""
        q = _as_rs(query)
        return _take_lists(lib().gth_mco_find(self._h, q._h, self._m(min_overlap)))

    def find_overlaps_regions(self, query, min_overlap=None):
        q = _as_rs(query)
        src = list(self._src)
        return [[Region(q[i].chr, src[v].start, src[v].end) for v in hits]
                for i, hits in enumerate(self.find_overlaps(q, min_overlap))]

    def subset_by(self, query, min_overlap=None):
        q = _as_rs(query)  # keep the temporary alive across the call
        h = lib().gth_mco_subset_by(self._h, q._h, self._m(min_overlap))
        if not h:
            _fail()
        return RegionSet._wrap(h)

    # ---- a batch of BED files in one device pass: element f equals the method above on RegionSet(paths[f]) ----------------
    def _bed_files(self, paths, mode, min_overlap):
        enc, arr = _paths_arg(paths)
        return _take_overlaps(lib().gth_mco_overlaps_bed_files(self._h, len(enc), arr, mode, self._m(min_overlap)))

    def count_overlaps_bed_files(self, paths, min_overlap=None):
        """Per file a uint32 array: count_overlaps(RegionSet(path)), every file parsed, sorted and counted on the device."""
        fq, _, vals, _ = self._bed_files(paths, _OVERLAPS_COUNT, min_overlap)
        return _per_file(vals, fq)

    def any_overlaps_bed_files(self, paths, min_overlap=None):
        """Per file a bool array: any_overlaps(RegionSet(path))."""
        fq, _, _, flags = self._bed_files(paths, _OVERLAPS_ANY, min_overlap)
        return _per_file(flags.astype(bool), fq)

    def find_overlaps_bed_files(self, paths, min_overlap=None):
        """Per file (offsets, vals): query i of RegionSet(path) hits vals[offsets[i]:offsets[i + 1]], in find_overlaps' order."""
        fq, off, vals, _ = self._bed_files(paths, _OVERLAPS_FIND, min_overlap)
        return _per_file_hits(fq, off, vals)

    def subset_by_bed_files(self, paths, min_overlap=None):
        """Per file subset_by(RegionSet(path)), the distinct hit regions reduced on the device."""
        return _subset_sets(lib().gth_mco_subset_by_bed_files, self._h, paths, self._m(min_overlap))


def parse_bed_file(path, chrom_names):
    """RegionSet::try_from's parse + sort run on the device: (chr ids, starts, ends) as uint32 arrays, ids index
    `chrom_names` (0xFFFFFFFF = a name that is not listed; those regions sort last)."""
    names = [n.encode() for n in chrom_names]
    arr = (C.c_char_p * max(len(names), 1))(*names)
    c, s, e = _take_lists(lib().gth_parse_bed_file(device(), os.fsencode(path), len(names), arr))
    return np.asarray(c, dtype=np.uint32), np.asarray(s, dtype=np.uint32), np.asarray(e, dtype=np.uint32)


def write_tokens_to_gtok(path, tokens):
    """gtars_io::write_tokens_to_gtok (gtok.rs:126-163)."""
    a = np.ascontiguousarray(tokens, dtype=np.uint32)
    if lib().gth_gtok_write(os.fsencode(path), len(a), a.ctypes.data, 0):
        _fail()


def append_tokens_to_gtok_file(path, tokens):
    a = np.ascontiguousarray(tokens, dtype=np.uint32)
    if lib().gth_gtok_write(os.fsencode(path), len(a), a.ctypes.data, 1):
        _fail()


def init_gtok_file(path):
    if lib().gth_gtok_write(os.fsencode(path), 0, None, 2):
        _fail()


def read_tokens_from_gtok(path):
    return _take_lists(lib().gth_gtok_read(os.fsencode(path)))[0]


class IndexedRegionSet:
    """gtars_overlaprs::IndexedRegionSet (indexed_region_set.rs): a RegionSet with its overlap index."""

    def __init__(self, regions, kind=AILIST):
        self._src = _as_rs(regions)
        self._h = lib().gth_irs_new(device(), self._src._h, kind)
        if not self._h:
            _fail()

    def __del__(self):
        if getattr(self, "_h", None):
            lib().gth_irs_free(self._h)
            self._h = None

    def regions(self):
        return self._src

    def find_overlaps(self, query, min_overlap=None):
        """Per query region: sorted, de-duplicated indices into the source set."""
        q = _as_rs(query)
        return _take_lists(lib().gth_irs_find(self._h, q._h, MultiChromOverlapper._m(min_overlap)))

    def subset_by_overlaps(self, query, min_overlap=None):
        q = _as_rs(query)
        h = lib().gth_irs_subset_by_overlaps(self._h, q._h, MultiChromOverlapper._m(min_overlap))
        if not h:
            _fail()
        return RegionSet._wrap(h)

    def intersect_all(self, query):
        return self.subset_by_overlaps(query, None)

    def find_overlaps_bed_files(self, paths, min_overlap=None):
        """Per file (offsets, vals): find_overlaps(RegionSet(path)) flattened, every query's indices sorted and de-duplicated."""
        enc, arr = _paths_arg(paths)
        fq, off, vals, _ = _take_overlaps(lib().gth_irs_find_bed_files(self._h, len(enc), arr, MultiChromOverlapper._m(min_overlap)))
        return _per_file_hits(fq, off, vals)

    def subset_by_overlaps_bed_files(self, paths, min_overlap=None):
        """Per file subset_by_overlaps(RegionSet(path))."""
        return _subset_sets(lib().gth_irs_subset_by_overlaps_bed_files, self._h, paths, MultiChromOverlapper._m(min_overlap))

    def count_overlaps(self, query, min_overlap=None):
        q = _as_rs(query)
        out = np.zeros(len(q), dtype=np.uint64)
        if lib().gth_irs_count(self._h, q._h, MultiChromOverlapper._m(min_overlap), out.ctypes.data):
            _fail()
        return [int(x) for x in out]

    def any_overlaps(self, query, min_overlap=None):
        q = _as_rs(query)
        out = np.zeros(len(q), dtype=np.uint8)
        if lib().gth_irs_any(self._h, q._h, MultiChromOverlapper._m(min_overlap), out.ctypes.data):
            _fail()
        return [bool(x) for x in out]


SCORING_ATAC, SCORING_CHIP = 0, 1


class ConsensusSet:
    """gtars_scoring::ConsensusSet (files.rs:60-99): consensus peaks, one column of the count matrix each."""

    def __init__(self, path):
        self._h = lib().gth_consensus_new(device(), os.fsencode(path))
        if not self._h:
            _fail()

    def __del__(self):
        if getattr(self, "_h", None):
            lib().gth_consensus_free(self._h)
            self._h = None

    def __len__(self):
        return int(lib().gth_consensus_len(self._h))


def region_scoring_from_fragments(fragment_files, consensus, mode=SCORING_ATAC, device_parse: bool = False):
    """gtars_scoring::region_scoring_from_fragments: uint32 [n_files, len(consensus)] (files in the given order).
    device_parse=True parses every file's text on the device (gtgpu_score_matrix_text / _gz), any file size."""
    files = [os.fsencode(p) for p in fragment_files]
    arr = (C.c_char_p * max(len(files), 1))(*files)
    out = np.zeros((len(files), len(consensus)), dtype=np.uint32)
    fn = lib().gth_region_scoring_device if device_parse else lib().gth_region_scoring
    if fn(consensus._h, len(files), arr, mode, out.ctypes.data):
        _fail()
    return out


def barcode_scoring_from_fragments(fragment_file, consensus, device_parse: bool = False):
    """gtars_scoring::barcode_scoring_from_fragments: {barcode: {peak index: count}}, barcodes in first-appearance order.
    device_parse=True parses the text and numbers the barcodes on the device (gtgpu_score_barcodes_text / _gz)."""
    fn = lib().gth_barcode_scoring_device if device_parse else lib().gth_barcode_scoring
    named = _take_lists(fn(consensus._h, os.fsencode(fragment_file)), named=True)
    return {bc: dict(zip(flat[0::2], flat[1::2])) for bc, flat in named}


class Tokenizer:
    """gtars.tokenizers.Tokenizer (gtars-tokenizers/src/tokenizer.rs)."""

    def __init__(self, path, _how=0):
        self._h = lib().gth_tokenizer_new(device(), os.fsencode(path), _how)
        if not self._h:
            _fail()

    @classmethod
    def from_bed(cls, path):
        return cls(path, 1)

    @classmethod
    def from_config(cls, path):
        return cls(path, 2)

    @classmethod
    def from_auto(cls, path):
        return cls(path, 0)

    def __del__(self):
        if getattr(self, "_h", None):
            lib().gth_tokenizer_free(self._h)
            self._h = None

    def get_vocab_size(self):
        return lib().gth_tokenizer_vocab_size(self._h)

    def __len__(self):
        return self.get_vocab_size()

    def convert_token_to_id(self, token):
        r = lib().gth_tokenizer_token_to_id(self._h, token.encode())
        return None if r < 0 else int(r)

    def convert_id_to_token(self, i):
        r = lib().gth_tokenizer_id_to_token(self._h, i)
        return None if r is None else r.decode()

    def _special(self, k):
        return lib().gth_tokenizer_special(self._h, k).decode()

    unk_token = property(lambda self: self._special(0))
    pad_token = property(lambda self: self._special(1))
    mask_token = property(lambda self: self._special(2))
    cls_token = property(lambda self: self._special(3))
    eos_token = property(lambda self: self._special(4))
    bos_token = property(lambda self: self._special(5))
    sep_token = property(lambda self: self._special(6))
    unk_token_id = property(lambda self: self.convert_token_to_id(self.unk_token))

    @staticmethod
    def _parse(regions):
        """A path, "chr:start-end" string(s), Region(s) or a RegionSet (extract_regions_from_py_any,
        gtars-python/src/utils/mod.rs:10-70)."""
        if isinstance(regions, RegionSet):
            return regions
        if isinstance(regions, (str, os.PathLike)) and os.path.exists(regions):
            return RegionSet(regions)
        if isinstance(regions, (str, Region)):
            regions = [regions]
        out = []
        for r in regions:
            if isinstance(r, str):
                c, rest = r.split(":")
                s, e = rest.split("-")
                out.append((c, int(s), int(e)))
            else:
                out.append(r)
        return RegionSet(out)

    def encode_bed_file(self, path):
        """encode(RegionSet(path)) with the BED text parsed, sorted and tokenized on the device."""
        return _take_lists(lib().gth_tokenizer_encode_bed_file(self._h, os.fsencode(path)))[0]

    def encode_bed_files(self, paths):
        """[encode_bed_file(p) for p in paths] in one device pass over all the files' text, of any total size
        (gtgpu_tokenize_bed_files; when every path ends in .gz the gzip bytes are inflated on the device too)."""
        paths = [os.fsencode(p) for p in paths]
        return _take_lists(lib().gth_tokenizer_encode_bed_files(self._h, len(paths), (C.c_char_p * max(len(paths), 1))(*paths)))

    def encode_batch(self, batches):
        """One Tokenizer::encode per element, all resolved in a single device pass."""
        sets = [self._parse(b) for b in batches]
        arr = (C.c_void_p * max(len(sets), 1))(*[s._h for s in sets])
        return _take_lists(lib().gth_tokenizer_encode_batch(self._h, len(sets), arr))

    def encode(self, regions):
        return self.encode_batch([regions])[0]

    def tokenize(self, regions):
        # tokenize() strings round-trip to encode() ids through first-appearance tokens (tokenizer.rs:140-171)
        return [self._first_token(i) for i in self.encode(regions)]

    def _first_token(self, i):
        tok = self.convert_id_to_token(i)
        return tok if self.convert_token_to_id(tok) == i else next(
            t for t in (self.convert_id_to_token(j) for j in range(self.get_vocab_size())) if self.convert_token_to_id(t) == i)

    def decode(self, ids):
        return [self.convert_id_to_token(i) or self.unk_token for i in ids]

    def __call__(self, regions):
        ids = self.encode(regions)
        return {"input_ids": ids, "attention_mask": [1] * len(ids)}


def tokenize_fragment_file(path, tokenizer: Tokenizer, device_parse: bool = False) -> dict:
    """gtars.tokenizers.tokenize_fragment_file (gtars-tokenizers/src/utils/fragments.rs:61-82): barcode -> token ids.
    device_parse=True also parses the text and numbers the barcodes on the device (gtgpu_tokenize_fragments_file / _gz),
    for a file of any size."""
    fn = lib().gth_tokenizer_fragments_device if device_parse else lib().gth_tokenizer_fragments
    return dict(_take_lists(fn(tokenizer._h, os.fsencode(path)), named=True))


def count_fragments_by_barcode(path, tokenizer: Tokenizer, device_parse: bool = False) -> dict:
    """gtars-tokenizers count_fragments_by_barcode (utils/fragments.rs:87-112): {barcode: {token id: count}}, barcodes in
    first-appearance order; a fragment with no hit counts under the unk id.  device_parse=True parses the text, tokenizes and
    counts on the device (gtgpu_count_fragments_file / _gz), for a file of any size."""
    fn = lib().gth_tokenizer_count_fragments_device if device_parse else lib().gth_tokenizer_count_fragments
    named = _take_lists(fn(tokenizer._h, os.fsencode(path)), named=True)
    return {bc: dict(zip(flat[0::2], flat[1::2])) for bc, flat in named}


class Igd:
    """gtars_igd::Igd built from region sets (Igd::from_named_region_sets, igd.rs:285-317)."""

    def __init__(self, region_sets):
        self._sets = [_as_rs(s) for s in region_sets]
        arr = (C.c_void_p * max(len(self._sets), 1))(*[s._h for s in self._sets])
        self._h = lib().gth_igd_new(device(), len(self._sets), arr)
        if not self._h:
            _fail()

    def __del__(self):
        if getattr(self, "_h", None):
            lib().gth_igd_free(self._h)
            self._h = None

    def save(self, path, names=None):
        """Igd::save (igd.rs:418-486): `path` (.igd) plus the companion .tsv, byte-for-byte the reference's files, written from
        the database on the device (gtgpu_igd_serialize) however it was built.  names[f] names file f in the .tsv (default
        set{f}).  A from_single_region_set Igd has no database to save and raises GtarsError."""
        names = list(names) if names is not None else [f"set{i}" for i in range(self.num_files())]
        nm = (C.c_char_p * max(len(names), 1))(*[n.encode() for n in names])
        if lib().gth_igd_save(self._h, len(names), nm, os.fsencode(path)):
            _fail()

    @classmethod
    def from_igd_file(cls, path):
        """Igd::from_igd_file (igd.rs:320-414): an existing .igd database straight into the device layout."""
        obj = cls.__new__(cls)
        obj._sets = []
        obj._h = lib().gth_igd_from_file(device(), os.fsencode(path))
        if not obj._h:
            _fail()
        return obj

    @classmethod
    def from_bed_files(cls, paths):
        """Igd([RegionSet(p) for p in paths]) with the files' text parsed on the device, their regions never on the host
        (gtgpu_igd_build_bed; when every path ends in .gz the gzip bytes are inflated on the device too)."""
        paths = [os.fsencode(p) for p in paths]
        obj = cls.__new__(cls)
        obj._sets = []
        obj._h = lib().gth_igd_from_bed_files(device(), len(paths), (C.c_char_p * max(len(paths), 1))(*paths))
        if not obj._h:
            _fail()
        return obj

    def info(self) -> dict:
        """gtgpu_igd_info of a database Igd: files, records kept, device bytes, LUT shift."""
        a = np.zeros(4, dtype=np.uint64)
        if lib().gth_igd_info(self._h, a.ctypes.data):
            _fail()
        return dict(n_files=int(a[0]), n_records=int(a[1]), device_bytes=int(a[2]), lut_shift=int(a[3]))

    @classmethod
    def from_single_region_set(cls, subject):
        """Igd::from_single_region_set (igd.rs:609-634): the subject side of two-set overlap queries."""
        obj = cls.__new__(cls)
        obj._sets = [_as_rs(subject)]
        obj._h = lib().gth_igd_single(device(), obj._sets[0]._h)
        if not obj._h:
            _fail()
        return obj

    def find_overlaps_regionset(self, query, min_overlap=1):
        """igd.rs:645-678: sorted (query idx, subject idx) pairs."""
        q = _as_rs(query)
        flat = _take_lists(lib().gth_igd_find_pairs(self._h, q._h, min_overlap))[0]
        return list(zip(flat[0::2], flat[1::2]))

    def count_overlaps_per_query(self, query, min_overlap=1):
        """igd.rs:690-722: distinct subject regions overlapping each query region."""
        q = _as_rs(query)
        return _take_lists(lib().gth_igd_count_per_query(self._h, q._h, min_overlap))[0]

    def num_files(self):
        return lib().gth_igd_num_files(self._h)

    def _count(self, sets, min_overlap, pairwise):
        sets = [_as_rs(s) for s in sets]
        arr = (C.c_void_p * max(len(sets), 1))(*[s._h for s in sets])
        out = np.zeros((len(sets), self.num_files()), dtype=np.uint64)
        if lib().gth_igd_count(self._h, len(sets), arr, min_overlap, 1 if pairwise else 0, out.ctypes.data):
            _fail()
        return out

    def count_set_overlaps(self, regions, min_overlap=1):
        return [int(x) for x in self._count([regions], min_overlap, True)[0]]

    def count_region_hits(self, regions, min_overlap=1):
        return [int(x) for x in self._count([regions], min_overlap, False)[0]]

    def count_bed_files(self, paths, min_overlap=1, pairwise=False) -> np.ndarray:
        """count_region_hits (pairwise: count_set_overlaps) of every BED file of `paths` as one query set, the files' text
        parsed on the device (gtgpu_igd_count_bed; the gzip bytes inflated there when every path ends in .gz): uint64
        [len(paths), num_files()], row i == count_region_hits(RegionSet(paths[i]))."""
        paths = [os.fsencode(p) for p in paths]
        out = np.zeros((len(paths), self.num_files()), dtype=np.uint64)
        regions = np.zeros(len(paths), dtype=np.uint64)
        if lib().gth_igd_count_bed_files(self._h, len(paths), (C.c_char_p * max(len(paths), 1))(*paths), min_overlap,
                                         1 if pairwise else 0, out.ctypes.data, regions.ctypes.data):
            _fail()
        return out


def write_igd_file(region_sets, names, path):
    """Igd::from_named_region_sets + Igd::save (igd.rs:285-317, 418-486) without building a device index: `path`
    (.igd) and the companion .tsv, byte for byte what the reference writes.  Host-only."""
    sets = [_as_rs(s) for s in region_sets]
    arr = (C.c_void_p * max(len(sets), 1))(*[s._h for s in sets])
    nm = (C.c_char_p * max(len(names), 1))(*[n.encode() for n in names])
    if lib().gth_igd_save_sets(len(sets), arr, nm, os.fsencode(path)):
        _fail()


def lola_contingency(igd: Igd, user_sets, universe, min_overlap=1) -> np.ndarray:
    """run_lola up to the 2x2 tables (gtars-lola/src/enrichment.rs:198-220): int64 [n_user, n_db, 4] = a, b, c, d."""
    sets = [_as_rs(s) for s in user_sets]
    uni = _as_rs(universe)
    arr = (C.c_void_p * max(len(sets), 1))(*[s._h for s in sets])
    out = np.zeros((len(sets), igd.num_files(), 4), dtype=np.int64)
    if lib().gth_lola_contingency(igd._h, len(sets), arr, uni._h, min_overlap, out.ctypes.data):
        _fail()
    return out


def lola_contingency_from_bed_files(igd: Igd, user_set_paths, universe_path, min_overlap=1) -> np.ndarray:
    """lola_contingency(igd, [RegionSet(p) for p in user_set_paths], RegionSet(universe_path)) with the user sets and the
    universe parsed on the device in one pass (gtgpu_igd_count_bed): int64 [n_user, n_db, 4] = a, b, c, d."""
    paths = [os.fsencode(p) for p in user_set_paths]
    out = np.zeros((len(paths), igd.num_files(), 4), dtype=np.int64)
    if lib().gth_lola_contingency_bed_files(igd._h, len(paths), (C.c_char_p * max(len(paths), 1))(*paths),
                                            os.fsencode(universe_path), min_overlap, out.ctypes.data):
        _fail()
    return out
