"""ctypes binding of include/gtars_gpu.h (libgtars_gpu.so) — flat arrays in, flat arrays out.

This is the same call surface a Rust `gtars-overlaprs-sys` crate would bind (INTEGRATION.md).  There is no CPU
fallback: if the shared library is missing or no CUDA device is usable, everything here raises.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_PKG = os.path.dirname(os.path.abspath(__file__))
# GTGPU_LIB selects an experimental build of the same library (tuning sweeps); the default is the in-tree product.
LIB_PATH = os.environ.get("GTGPU_LIB") or os.path.join(_PKG, "libgtars_gpu.so")

SCORE_ATAC, SCORE_CHIP = 0, 1
OVERLAPS_COUNT, OVERLAPS_ANY, OVERLAPS_FIND, OVERLAPS_SUBSET = 0, 1, 2, 3
KIND_BITS, KIND_AILIST = 0, 1
UNKNOWN_CHROM = 0xFFFFFFFF

# every symbol include/gtars_gpu.h declares: name -> (restype, argtypes)
_vp, _u32, _u64, _i32 = C.c_void_p, C.c_uint32, C.c_uint64, C.c_int32
SIGNATURES = {
    "gtgpu_last_error": (C.c_char_p, []),
    "gtgpu_version": (C.c_char_p, []),
    "gtgpu_device_count": (_i32, [_vp]),
    "gtgpu_init": (_i32, [_i32, _vp, _vp]),
    "gtgpu_init_multi": (_i32, [_i32, _vp, _vp]),
    "gtgpu_ctx_devices": (_i32, [_vp, _vp, _vp, _i32]),
    "gtgpu_shutdown": (_i32, [_vp]),
    "gtgpu_synchronize": (_i32, [_vp]),
    "gtgpu_launch_count": (_i32, [_vp, _vp]),
    "gtgpu_timing_enable": (_i32, [_vp, _i32]),
    "gtgpu_timing_read": (_i32, [_vp, _vp, _u32, _vp]),
    "gtgpu_host_alloc": (_i32, [_u64, _vp]),
    "gtgpu_host_free": (_i32, [_vp]),
    "gtgpu_buf_data": (_vp, [_vp]),
    "gtgpu_buf_len": (_u64, [_vp]),
    "gtgpu_buf_free": (_i32, [_vp]),
    "gtgpu_index_build": (_i32, [_vp, _i32, _u32, _vp, _vp, _vp, _vp, _vp]),
    "gtgpu_index_free": (_i32, [_vp]),
    "gtgpu_index_info": (_i32, [_vp, _vp]),
    "gtgpu_count": (_i32, [_vp, _u64, _vp, _vp, _vp, _i32, _vp]),
    "gtgpu_bits_count": (_i32, [_vp, _u64, _vp, _vp, _vp, _vp]),
    "gtgpu_any": (_i32, [_vp, _u64, _vp, _vp, _vp, _i32, _vp]),
    "gtgpu_find": (_i32, [_vp, _u64, _vp, _vp, _vp, _i32, _vp, _vp]),
    "gtgpu_tokenize_files": (_i32, [_vp, _u64, _vp, _vp, _vp, _vp, _u32, _vp, _vp]),
    "gtgpu_tokenize_files_runs": (_i32, [_vp, _u64, _vp, _u64, _vp, _vp, _vp, _vp, _u32, _vp, _vp]),
    "gtgpu_tokenize_files_compact": (_i32, [_vp, _u64, _vp, _u64, _vp, _vp, _vp, _vp, _u64, _vp, _vp, _u32, _vp, _vp]),
    "gtgpu_marshal_compact": (_i32, [_u64, _vp, _vp, _vp, _u64, _vp, _i32, _vp, _u64, _vp, _vp, _vp, _u64, _vp, _vp, _vp]),
    "gtgpu_tokenize_files_packed": (_i32, [_vp, _u64, _vp, _u64, _vp, _vp, _u32, _vp, _vp, _u64, _vp, _vp, _vp, _u32, _vp, _vp]),
    "gtgpu_marshal_packed": (_i32, [_u64, _vp, _vp, _vp, _u64, _vp, _i32, _u32, _vp, _vp, _u64, _vp, _vp, _vp, _u64, _vp, _vp, _vp, _vp,
                                    _vp]),
    "gtgpu_tokenize_fragments": (_i32, [_vp, _u64, _vp, _vp, _vp, _vp, _u32, _u32, _vp, _vp]),
    "gtgpu_tokenize_fragments_dev": (_i32, [_vp, _u64, _vp, _vp, _vp, _vp, _u32, _u32, _vp, _vp, _u64, _vp]),
    "gtgpu_parse_bed": (_i32, [_vp, _vp, _u64, _u32, _vp, _vp, _vp, _vp, _vp, _vp]),
    "gtgpu_tokenize_bed": (_i32, [_vp, _vp, _u64, _u32, _vp, _vp, _u32, _vp]),
    "gtgpu_tokenize_bed_files": (_i32, [_vp, _u64, _vp, _vp, _u32, _vp, _vp, _u32, _vp, _vp]),
    "gtgpu_tokenize_bed_files_gz": (_i32, [_vp, _u64, _vp, _u64, _vp, _vp, _u32, _vp, _vp, _u32, _vp, _vp]),
    "gtgpu_overlaps_bed_files": (_i32, [_vp, _i32, _u64, _vp, _vp, _u32, _vp, _vp, _i32, _u64, _vp, _vp, _vp, _vp]),
    "gtgpu_overlaps_bed_files_gz": (_i32, [_vp, _i32, _u64, _vp, _u64, _vp, _vp, _u32, _vp, _vp, _i32, _u64, _vp, _vp, _vp, _vp]),
    "gtgpu_tokenize_fragments_text": (_i32, [_vp, _vp, _u64, _u32, _vp, _vp, _u32, _vp, _vp, _vp, _vp]),
    "gtgpu_gzip_members": (_i32, [_vp, _u64, _u64, _vp, _vp]),
    "gtgpu_gunzip": (_i32, [_vp, _u64, _vp, _vp, _vp, _vp]),
    "gtgpu_tokenize_bed_gz": (_i32, [_vp, _u64, _vp, _vp, _u32, _vp, _vp, _u32, _vp]),
    "gtgpu_tokenize_fragments_gz": (_i32, [_vp, _u64, _vp, _vp, _u32, _vp, _vp, _u32, _vp, _vp, _vp, _vp, _vp]),
    "gtgpu_tokenize_fragments_file": (_i32, [_vp, _vp, _u64, _u32, _vp, _vp, _u32, _vp, _vp, _vp, _vp, _vp]),
    "gtgpu_tokenize_fragments_file_gz": (_i32, [_vp, _u64, _vp, _vp, _u32, _vp, _vp, _u32, _vp, _vp, _vp, _vp, _vp]),
    "gtgpu_count_fragments_file": (_i32, [_vp, _vp, _u64, _u32, _vp, _vp, _u32, _vp, _vp, _vp, _vp, _vp, _vp]),
    "gtgpu_count_fragments_file_gz": (_i32, [_vp, _u64, _vp, _vp, _u32, _vp, _vp, _u32, _vp, _vp, _vp, _vp, _vp, _vp]),
    "gtgpu_score_matrix": (_i32, [_vp, _u64, _vp, _u64, _vp, _vp, _vp, _i32, _u64, _vp]),
    "gtgpu_score_matrix_dev": (_i32, [_vp, _u64, _vp, _u64, _vp, _vp, _vp, _i32, _u64, _vp]),
    "gtgpu_score_barcodes": (_i32, [_vp, _u64, _vp, _vp, _vp, _vp, _u32, _vp, _vp, _vp]),
    "gtgpu_score_matrix_text": (_i32, [_vp, _vp, _u64, _u32, _vp, _vp, _i32, _u64, _vp]),
    "gtgpu_score_matrix_gz": (_i32, [_vp, _u64, _vp, _vp, _u32, _vp, _vp, _i32, _u64, _vp]),
    "gtgpu_score_barcodes_text": (_i32, [_vp, _vp, _u64, _u32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "gtgpu_score_barcodes_gz": (_i32, [_vp, _u64, _vp, _vp, _u32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "gtgpu_igd_build": (_i32, [_vp, _u64, _vp, _u32, _vp, _vp, _vp, _vp]),
    "gtgpu_igd_build_bed": (_i32, [_vp, _u64, _vp, _vp, _vp, _vp, _vp, _vp]),
    "gtgpu_igd_build_bed_gz": (_i32, [_vp, _u64, _vp, _u64, _vp, _vp, _vp, _vp, _vp, _vp]),
    "gtgpu_igd_free": (_i32, [_vp]),
    "gtgpu_igd_serialize": (_i32, [_vp, _u32, _vp, _vp, _vp, _vp, _vp]),
    "gtgpu_igd_info": (_i32, [_vp, _vp]),
    "gtgpu_igd_count_set_overlaps": (_i32, [_vp, _u64, _vp, _vp, _vp, _vp, _i32, _vp]),
    "gtgpu_igd_count_region_hits": (_i32, [_vp, _u64, _vp, _vp, _vp, _vp, _i32, _vp]),
    "gtgpu_igd_count_dev": (_i32, [_vp, _i32, _u64, _vp, _vp, _vp, _vp, _i32, _vp]),
    "gtgpu_igd_count_bed": (_i32, [_vp, _i32, _u64, _vp, _vp, _u32, _vp, _vp, _i32, _vp, _vp]),
    "gtgpu_igd_count_bed_gz": (_i32, [_vp, _i32, _u64, _vp, _u64, _vp, _vp, _u32, _vp, _vp, _i32, _vp, _vp]),
    "gtgpu_comm_unique_id": (_i32, [_vp]),
    "gtgpu_comm_init": (_i32, [_vp, _i32, _i32, _vp]),
    "gtgpu_comm_free": (_i32, [_vp]),
    "gtgpu_igd_count_sharded": (_i32, [_vp, _vp, _i32, _u64, _u64, _vp, _vp, _vp, _vp, _i32, _vp]),
    "gtgpu_count_dev": (_i32, [_vp, _u64, _vp, _vp, _vp, _i32, _vp]),
    "gtgpu_find_dev": (_i32, [_vp, _u64, _vp, _vp, _vp, _i32, _u64, _vp, _vp, _u64, _vp, _vp, _vp]),
    "gtgpu_unk_rule_dev": (_i32, [_vp, _u64, _vp, _vp, _u32, _vp, _vp, _vp]),
}


class GtarsGpuError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"gtars_gpu error {code}: {msg}")
        self.code = code


_lib = None


def lib():
    """Load libgtars_gpu.so (built by __graft_entry__.build() / `make -C gtars_b200/csrc`)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(f"{LIB_PATH} is missing: build it with `make -C gtars_b200/csrc` "
                              "(there is no CPU fallback)")
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def check(status):
    if status != 0:
        raise GtarsGpuError(status, lib().gtgpu_last_error().decode(errors="replace"))


def _arr(a, dtype):
    return np.ascontiguousarray(a, dtype=dtype)


def _p(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


def device_count() -> int:
    n = C.c_int32(0)
    check(lib().gtgpu_device_count(C.byref(n)))
    return n.value


def pinned_empty(n, dtype) -> np.ndarray:
    """numpy array backed by pinned host memory (gtgpu_host_alloc); freed when the array is collected."""
    dtype = np.dtype(dtype)
    ptr = C.c_void_p()
    check(lib().gtgpu_host_alloc(max(int(n) * dtype.itemsize, 64), C.byref(ptr)))
    buf = (C.c_char * max(int(n) * dtype.itemsize, 1)).from_address(ptr.value)
    arr = np.frombuffer(buf, dtype=dtype, count=int(n))

    class _Owner:
        def __init__(self, p):
            self.p = p

        def __del__(self):
            try:
                lib().gtgpu_host_free(self.p)
            except Exception:
                pass

    _OWNERS[ptr.value] = _Owner(ptr.value)
    return arr


_OWNERS = {}


def pinned_free(arr: np.ndarray):
    o = _OWNERS.pop(arr.ctypes.data, None)
    if o is not None:
        lib().gtgpu_host_free(o.p)
        o.p = None


def _take(buf_handle, dtype=np.uint32, copy=True) -> np.ndarray:
    L = lib()
    n = L.gtgpu_buf_len(buf_handle)
    out = np.empty(n, dtype=dtype)
    if n:
        C.memmove(out.ctypes.data, L.gtgpu_buf_data(buf_handle), n * out.itemsize)
    L.gtgpu_buf_free(buf_handle)
    return out


class Context:
    """gtgpu_ctx: one device (`device`, optionally on the caller's `stream`) or, with `devices=[...]`, one context over
    several devices of this process (gtgpu_init_multi) whose entry points shard their work internally."""

    def __init__(self, device: int = 0, stream: int | None = None, devices=None):
        self._h = C.c_void_p()
        if devices is not None:
            ids = np.ascontiguousarray(devices, dtype=np.int32)
            check(lib().gtgpu_init_multi(len(ids), _p(ids), C.byref(self._h)))
            self.device = int(ids[0])
        else:
            check(lib().gtgpu_init(device, C.c_void_p(stream) if stream else None, C.byref(self._h)))
            self.device = device

    def devices(self):
        n = C.c_int32(0)
        ids = np.zeros(64, dtype=np.int32)
        check(lib().gtgpu_ctx_devices(self._h, C.byref(n), _p(ids), 64))
        return [int(x) for x in ids[:n.value]]

    def close(self):
        if getattr(self, "_h", None):
            lib().gtgpu_shutdown(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def synchronize(self):
        check(lib().gtgpu_synchronize(self._h))

    def launch_count(self) -> int:
        n = C.c_uint64(0)
        check(lib().gtgpu_launch_count(self._h, C.byref(n)))
        return n.value

    def timing_enable(self, on=True):
        check(lib().gtgpu_timing_enable(self._h, 1 if on else 0))

    def timing_read(self, cap=256):
        ms = (C.c_float * cap)()
        n = C.c_uint32(0)
        check(lib().gtgpu_timing_read(self._h, ms, cap, C.byref(n)))
        return [ms[i] for i in range(min(cap, n.value))]

    def unk_rule_dev(self, n_files, d_raw_tok, d_raw_ids, unk_id, d_out_tok, d_out_ids, d_n_empty):
        check(lib().gtgpu_unk_rule_dev(self._h, n_files, d_raw_tok, d_raw_ids, unk_id, d_out_tok, d_out_ids, d_n_empty))


class Index:
    """gtgpu_index: per-chromosome Bits / AIList on the device."""

    def __init__(self, ctx: Context, kind: int, chrom_offsets, starts, ends, vals=None):
        self.ctx = ctx
        self.kind = kind
        co = _arr(chrom_offsets, np.uint64)
        s, e = _arr(starts, np.uint32), _arr(ends, np.uint32)
        v = _arr(vals, np.uint32) if vals is not None else None
        if len(s) != len(e) or (v is not None and len(v) != len(s)) or (len(co) and int(co[-1]) != len(s)):
            raise ValueError("index arrays disagree in length")
        self.n_chroms = max(len(co) - 1, 0)
        self._h = C.c_void_p()
        check(lib().gtgpu_index_build(ctx._h, kind, self.n_chroms, _p(co), _p(s), _p(e), _p(v), C.byref(self._h)))

    def close(self):
        if getattr(self, "_h", None) and getattr(self.ctx, "_h", None):
            lib().gtgpu_index_free(self._h)
        self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def info(self) -> dict:
        a = (C.c_uint64 * 12)()
        check(lib().gtgpu_index_info(self._h, a))
        return dict(n_intervals=a[0], n_segments=a[1], device_bytes=a[2], lut_shift=a[3], max_components=a[4],
                    proper=bool(a[5]), bt_bins=a[6], bt_overflow_bins=a[7], bt_shift=a[8], bt_pool_windows=a[9],
                    lean_kernel=bool(a[10]), lean_fell_back=bool(a[11]))

    # ---- host-buffer entry points -------------------------------------------------------------------------------
    def count(self, chr, start, end, min_overlap=0) -> np.ndarray:
        chr, start, end = _arr(chr, np.uint32), _arr(start, np.uint32), _arr(end, np.uint32)
        out = np.empty(len(chr), dtype=np.uint32)
        check(lib().gtgpu_count(self._h, len(chr), _p(chr), _p(start), _p(end), min_overlap, _p(out)))
        return out

    def bits_count(self, chr, start, end) -> np.ndarray:
        chr, start, end = _arr(chr, np.uint32), _arr(start, np.uint32), _arr(end, np.uint32)
        out = np.empty(len(chr), dtype=np.uint64)
        check(lib().gtgpu_bits_count(self._h, len(chr), _p(chr), _p(start), _p(end), _p(out)))
        return out

    def any(self, chr, start, end, min_overlap=0) -> np.ndarray:
        chr, start, end = _arr(chr, np.uint32), _arr(start, np.uint32), _arr(end, np.uint32)
        out = np.empty(len(chr), dtype=np.uint8)
        check(lib().gtgpu_any(self._h, len(chr), _p(chr), _p(start), _p(end), min_overlap, _p(out)))
        return out.astype(bool)

    def find(self, chr, start, end, min_overlap=0):
        chr, start, end = _arr(chr, np.uint32), _arr(start, np.uint32), _arr(end, np.uint32)
        off = np.empty(len(chr) + 1, dtype=np.uint64)
        h = C.c_void_p()
        check(lib().gtgpu_find(self._h, len(chr), _p(chr), _p(start), _p(end), min_overlap, _p(off), C.byref(h)))
        return off, _take(h)

    def tokenize_files(self, file_offsets, chr, start, end, unk_id, keep_buf=False):
        fo = _arr(file_offsets, np.uint64)
        chr, start, end = _arr(chr, np.uint32), _arr(start, np.uint32), _arr(end, np.uint32)
        out_off = np.empty(len(fo), dtype=np.uint64)
        h = C.c_void_p()
        check(lib().gtgpu_tokenize_files(self._h, len(fo) - 1, _p(fo), _p(chr), _p(start), _p(end), unk_id,
                                         _p(out_off), C.byref(h)))
        if keep_buf:
            return out_off, h
        return out_off, _take(h)

    def tokenize_files_runs(self, file_offsets, run_offsets, run_chr, start, end, unk_id, keep_buf=False):
        fo, ro = _arr(file_offsets, np.uint64), _arr(run_offsets, np.uint64)
        rc, start, end = _arr(run_chr, np.uint32), _arr(start, np.uint32), _arr(end, np.uint32)
        out_off = np.empty(len(fo), dtype=np.uint64)
        h = C.c_void_p()
        check(lib().gtgpu_tokenize_files_runs(self._h, len(fo) - 1, _p(fo), len(rc), _p(ro), _p(rc), _p(start), _p(end),
                                              unk_id, _p(out_off), C.byref(h)))
        if keep_buf:
            return out_off, h
        return out_off, _take(h)

    def tokenize_files_compact(self, file_offsets, run_offsets, run_chr, start, width16, wide_index, wide_end, unk_id,
                               keep_buf=False):
        fo, ro = _arr(file_offsets, np.uint64), _arr(run_offsets, np.uint64)
        rc, start, w16 = _arr(run_chr, np.uint32), _arr(start, np.uint32), _arr(width16, np.uint16)
        wi, we = _arr(wide_index, np.uint64), _arr(wide_end, np.uint32)
        out_off = np.empty(len(fo), dtype=np.uint64)
        h = C.c_void_p()
        check(lib().gtgpu_tokenize_files_compact(self._h, len(fo) - 1, _p(fo), len(rc), _p(ro), _p(rc), _p(start), _p(w16),
                                                 len(wi), _p(wi), _p(we), unk_id, _p(out_off), C.byref(h)))
        if keep_buf:
            return out_off, h
        return out_off, _take(h)

    def tokenize_files_packed(self, file_offsets, run_offsets, run_chr, width_bits, packed, anchors, exc_index, exc_start, exc_end,
                              unk_id, keep_buf=False):
        fo, ro = _arr(file_offsets, np.uint64), _arr(run_offsets, np.uint64)
        rc, pk, an = _arr(run_chr, np.uint32), _arr(packed, np.uint32), _arr(anchors, np.uint32)
        xi, xs, xe = _arr(exc_index, np.uint64), _arr(exc_start, np.uint32), _arr(exc_end, np.uint32)
        out_off = np.empty(len(fo), dtype=np.uint64)
        h = C.c_void_p()
        check(lib().gtgpu_tokenize_files_packed(self._h, len(fo) - 1, _p(fo), len(rc), _p(ro), _p(rc), width_bits, _p(pk), _p(an),
                                                len(xi), _p(xi), _p(xs), _p(xe), unk_id, _p(out_off), C.byref(h)))
        if keep_buf:
            return out_off, h
        return out_off, _take(h)

    def tokenize_fragments(self, chr, start, end, barcode, n_barcodes, unk_id, keep_buf=False):
        chr, start, end, barcode = (_arr(a, np.uint32) for a in (chr, start, end, barcode))
        out_off = np.empty(n_barcodes + 1, dtype=np.uint64)
        h = C.c_void_p()
        check(lib().gtgpu_tokenize_fragments(self._h, len(chr), _p(chr), _p(start), _p(end), _p(barcode), n_barcodes,
                                             unk_id, _p(out_off), C.byref(h)))
        if keep_buf:
            return out_off, h
        return out_off, _take(h)

    def tokenize_bed(self, text: bytes, chrom_names, unk_id):
        """gtgpu_tokenize_bed: BED text in, token ids out (parse + sort + encode on the device)."""
        blob = b"".join(n.encode() for n in chrom_names)
        offs = np.zeros(len(chrom_names) + 1, dtype=np.uint32)
        offs[1:] = np.cumsum([len(n.encode()) for n in chrom_names])
        h = C.c_void_p()
        check(lib().gtgpu_tokenize_bed(self._h, text, len(text), len(chrom_names), blob, _p(offs), unk_id, C.byref(h)))
        return _take(h)

    def tokenize_bed_gz(self, gz: bytes, chrom_names, unk_id, member_offsets=None):
        """gtgpu_tokenize_bed_gz: gzip members in, token ids out (inflate + parse + sort + encode on the device)."""
        mo = _arr(member_offsets if member_offsets is not None else gzip_members(gz), np.uint64)
        blob, offs = _names_blob(chrom_names)
        h = C.c_void_p()
        check(lib().gtgpu_tokenize_bed_gz(self._h, len(mo) - 1, gz, _p(mo), len(chrom_names), blob, _p(offs), unk_id, C.byref(h)))
        return _take(h)

    def tokenize_bed_files(self, text, file_offsets, chrom_names, unk_id):
        """gtgpu_tokenize_bed_files: file f = text[file_offsets[f]:file_offsets[f + 1]] parsed, sorted per file and tokenized on
        the device.  Returns (file_token_offsets, ids) as tokenize_files does.  `text` may be a uint8 numpy array."""
        fo = _arr(file_offsets, np.uint64)
        blob, offs = _names_blob(chrom_names)
        out_off = np.empty(len(fo), dtype=np.uint64)
        h = C.c_void_p()
        check(lib().gtgpu_tokenize_bed_files(self._h, len(fo) - 1, _text_ptr(text), _p(fo), len(chrom_names), blob, _p(offs), unk_id,
                                             _p(out_off), C.byref(h)))
        return out_off, _take(h)

    def tokenize_bed_files_gz(self, gz, file_members, member_offsets, chrom_names, unk_id):
        """gtgpu_tokenize_bed_files_gz: file f = gzip members [file_members[f], file_members[f + 1]) of `gz` (member_offsets as
        gzip_members returns them), inflated, parsed, sorted per file and tokenized on the device."""
        fm, mo = _arr(file_members, np.uint64), _arr(member_offsets, np.uint64)
        blob, offs = _names_blob(chrom_names)
        out_off = np.empty(len(fm), dtype=np.uint64)
        h = C.c_void_p()
        check(lib().gtgpu_tokenize_bed_files_gz(self._h, len(fm) - 1, _p(fm), len(mo) - 1, _text_ptr(gz), _p(mo), len(chrom_names),
                                                blob, _p(offs), unk_id, _p(out_off), C.byref(h)))
        return out_off, _take(h)

    def _overlaps_bed(self, mode, n_files, chrom_names, min_overlap, keys, call):
        blob, offs = _names_blob(chrom_names)
        k = None if keys is None else _arr(keys, np.uint32)
        fq = np.empty(n_files + 1, dtype=np.uint64)
        ho, hv = C.c_void_p(), C.c_void_p()
        check(call(blob, offs, min_overlap, 0 if k is None else len(k), _p(k), _p(fq), C.byref(ho), C.byref(hv)))
        vals = _take(hv, np.uint8 if mode == OVERLAPS_ANY else np.uint32)
        return fq, (_take(ho, np.uint64) if ho.value else None), vals

    def overlaps_bed_text(self, mode, text, file_offsets, chrom_names, min_overlap=0, keys=None):
        """gtgpu_overlaps_bed_files: file f = text[file_offsets[f]:file_offsets[f + 1]] parsed and sorted per file on the device,
        then counted / flagged / found / subset (mode OVERLAPS_*).  Returns (file_queries, offsets or None, values)."""
        fo = _arr(file_offsets, np.uint64)
        return self._overlaps_bed(mode, len(fo) - 1, chrom_names, min_overlap, keys, lambda blob, offs, m, nk, kp, fq, ho, hv:
                                  lib().gtgpu_overlaps_bed_files(self._h, mode, len(fo) - 1, _text_ptr(text), _p(fo), len(chrom_names),
                                                                 blob, _p(offs), m, nk, kp, fq, ho, hv))

    def overlaps_bed_gz(self, mode, gz, file_members, member_offsets, chrom_names, min_overlap=0, keys=None):
        """gtgpu_overlaps_bed_files_gz: file f = gzip members [file_members[f], file_members[f + 1]) of `gz`."""
        fm, mo = _arr(file_members, np.uint64), _arr(member_offsets, np.uint64)
        return self._overlaps_bed(mode, len(fm) - 1, chrom_names, min_overlap, keys, lambda blob, offs, m, nk, kp, fq, ho, hv:
                                  lib().gtgpu_overlaps_bed_files_gz(self._h, mode, len(fm) - 1, _p(fm), len(mo) - 1, _text_ptr(gz), _p(mo),
                                                                    len(chrom_names), blob, _p(offs), m, nk, kp, fq, ho, hv))

    def tokenize_fragments_text(self, text: bytes, chrom_names, unk_id, gz_member_offsets=None):
        """gtgpu_tokenize_fragments_text (or _gz when gz_member_offsets is given: `text` is then the gzip data):
        ([barcode strings], offsets, ids)."""
        blob, offs = _names_blob(chrom_names)
        nb = C.c_uint32(0)
        hs, ho, hi, ht = C.c_void_p(), C.c_void_p(), C.c_void_p(), C.c_void_p()
        if gz_member_offsets is not None:
            mo = _arr(gz_member_offsets, np.uint64)
            check(lib().gtgpu_tokenize_fragments_gz(self._h, len(mo) - 1, text, _p(mo), len(chrom_names), blob, _p(offs), unk_id,
                                                    C.byref(nb), C.byref(hs), C.byref(ho), C.byref(hi), C.byref(ht)))
            text = _take(ht, dtype=np.uint8).tobytes()
        else:
            check(lib().gtgpu_tokenize_fragments_text(self._h, text, len(text), len(chrom_names), blob, _p(offs), unk_id,
                                                      C.byref(nb), C.byref(hs), C.byref(ho), C.byref(hi)))
        spans = _take(hs).reshape(-1, 2)
        off = _take(ho, dtype=np.uint64)
        ids = _take(hi)
        return [text[int(a):int(a) + int(n)].decode() for a, n in spans[:nb.value]], off, ids

    def tokenize_fragments_file(self, text, chrom_names, unk_id, gz_member_offsets=None):
        """gtgpu_tokenize_fragments_file (or _gz when gz_member_offsets is given: `text` is then the gzip data), any size:
        ([barcode strings], offsets[n + 1], ids).  `text` may be a uint8 numpy array (a multi-GB text is not copied)."""
        blob, offs = _names_blob(chrom_names)
        nb = C.c_uint32(0)
        hn, hno, ho, hi = C.c_void_p(), C.c_void_p(), C.c_void_p(), C.c_void_p()
        outs = (C.byref(nb), C.byref(hn), C.byref(hno), C.byref(ho), C.byref(hi))
        if gz_member_offsets is not None:
            mo = _arr(gz_member_offsets, np.uint64)
            check(lib().gtgpu_tokenize_fragments_file_gz(self._h, len(mo) - 1, _text_ptr(text), _p(mo), len(chrom_names), blob, _p(offs),
                                                         unk_id, *outs))
        else:
            check(lib().gtgpu_tokenize_fragments_file(self._h, _text_ptr(text), _text_len(text), len(chrom_names), blob, _p(offs), unk_id,
                                                      *outs))
        names = _take(hn, dtype=np.uint8).tobytes()
        no = _take(hno, dtype=np.uint64)
        return [names[int(a):int(b)].decode() for a, b in zip(no[:-1], no[1:])], _take(ho, dtype=np.uint64), _take(hi)

    def count_fragments_file(self, text, chrom_names, unk_id, gz_member_offsets=None):
        """gtgpu_count_fragments_file (or _gz when gz_member_offsets is given: `text` is then the gzip data), any size:
        ([barcode strings], offsets[n + 1], tokens, counts); per barcode its distinct token ids ascending, with their counts."""
        blob, offs = _names_blob(chrom_names)
        nb = C.c_uint32(0)
        hn, hno, ho, ht, hc = C.c_void_p(), C.c_void_p(), C.c_void_p(), C.c_void_p(), C.c_void_p()
        outs = (C.byref(nb), C.byref(hn), C.byref(hno), C.byref(ho), C.byref(ht), C.byref(hc))
        if gz_member_offsets is not None:
            mo = _arr(gz_member_offsets, np.uint64)
            check(lib().gtgpu_count_fragments_file_gz(self._h, len(mo) - 1, _text_ptr(text), _p(mo), len(chrom_names), blob, _p(offs),
                                                      unk_id, *outs))
        else:
            check(lib().gtgpu_count_fragments_file(self._h, _text_ptr(text), _text_len(text), len(chrom_names), blob, _p(offs), unk_id,
                                                   *outs))
        names = _take(hn, dtype=np.uint8).tobytes()
        no = _take(hno, dtype=np.uint64)
        return ([names[int(a):int(b)].decode() for a, b in zip(no[:-1], no[1:])], _take(ho, dtype=np.uint64), _take(ht), _take(hc))

    def score_matrix(self, file_offsets, chr, start, end, mode, n_cols):
        """region_scoring_from_fragments: uint32 [n_files, n_cols]."""
        fo = _arr(file_offsets, np.uint64)
        chr, start, end = (_arr(a, np.uint32) for a in (chr, start, end))
        out = np.empty((len(fo) - 1, n_cols), dtype=np.uint32)
        check(lib().gtgpu_score_matrix(self._h, len(fo) - 1, _p(fo), len(chr), _p(chr), _p(start), _p(end), mode, n_cols, _p(out)))
        return out

    def score_matrix_dev(self, n_files, d_file_offsets, n, d_chr, d_start, d_end, mode, n_cols, d_out):
        check(lib().gtgpu_score_matrix_dev(self._h, n_files, d_file_offsets, n, d_chr, d_start, d_end, mode, n_cols, d_out))

    def score_barcodes(self, chr, start, end, barcode, n_barcodes):
        """barcode_scoring_from_fragments: (offsets[n_barcodes + 1], peaks, counts) sorted by (barcode, peak)."""
        chr, start, end, barcode = (_arr(a, np.uint32) for a in (chr, start, end, barcode))
        out_off = np.empty(n_barcodes + 1, dtype=np.uint64)
        hp, hc = C.c_void_p(), C.c_void_p()
        check(lib().gtgpu_score_barcodes(self._h, len(chr), _p(chr), _p(start), _p(end), _p(barcode), n_barcodes,
                                         _p(out_off), C.byref(hp), C.byref(hc)))
        return out_off, _take(hp), _take(hc)

    def score_matrix_text(self, text: bytes, chrom_names, mode, n_cols, gz_member_offsets=None):
        """gtgpu_score_matrix_text (or _gz when gz_member_offsets is given: `text` is then the gzip data): the file's
        uint32 row [n_cols] of region_scoring_from_fragments, parsed on the device."""
        blob, offs = _names_blob(chrom_names)
        out = np.empty(n_cols, dtype=np.uint32)
        if gz_member_offsets is not None:
            mo = _arr(gz_member_offsets, np.uint64)
            check(lib().gtgpu_score_matrix_gz(self._h, len(mo) - 1, text, _p(mo), len(chrom_names), blob, _p(offs), mode, n_cols,
                                              _p(out)))
        else:
            check(lib().gtgpu_score_matrix_text(self._h, _text_ptr(text), _text_len(text), len(chrom_names), blob, _p(offs), mode, n_cols,
                                                _p(out)))
        return out

    def score_barcodes_text(self, text: bytes, chrom_names, gz_member_offsets=None):
        """gtgpu_score_barcodes_text (or _gz): ([barcode strings], offsets[n + 1], peaks, counts) sorted by (barcode, peak)."""
        blob, offs = _names_blob(chrom_names)
        nb = C.c_uint32(0)
        hn, hno, ho, hp, hc = C.c_void_p(), C.c_void_p(), C.c_void_p(), C.c_void_p(), C.c_void_p()
        outs = (C.byref(nb), C.byref(hn), C.byref(hno), C.byref(ho), C.byref(hp), C.byref(hc))
        if gz_member_offsets is not None:
            mo = _arr(gz_member_offsets, np.uint64)
            check(lib().gtgpu_score_barcodes_gz(self._h, len(mo) - 1, text, _p(mo), len(chrom_names), blob, _p(offs), *outs))
        else:
            check(lib().gtgpu_score_barcodes_text(self._h, _text_ptr(text), _text_len(text), len(chrom_names), blob, _p(offs), *outs))
        names = _take(hn, dtype=np.uint8).tobytes()
        no = _take(hno, dtype=np.uint64)
        return ([names[int(a):int(b)].decode() for a, b in zip(no[:-1], no[1:])], _take(ho, dtype=np.uint64), _take(hp), _take(hc))

    # ---- device-resident entry points (raw device pointers as ints) ----------------------------------------------------
    def count_dev(self, n, d_chr, d_start, d_end, min_overlap, d_out):
        check(lib().gtgpu_count_dev(self._h, n, d_chr, d_start, d_end, min_overlap, d_out))

    def tokenize_fragments_dev(self, n, d_chr, d_start, d_end, d_barcode, n_barcodes, unk_id, d_out_barcode_offsets, d_out_ids,
                               ids_capacity, d_out_total):
        check(lib().gtgpu_tokenize_fragments_dev(self._h, n, d_chr, d_start, d_end, d_barcode, n_barcodes, unk_id,
                                                 d_out_barcode_offsets, d_out_ids, ids_capacity, d_out_total))

    def find_dev(self, n, d_chr, d_start, d_end, min_overlap, n_files, d_file_offsets, d_out_ids, ids_capacity,
                 d_out_offsets, d_out_file_tok, d_out_total):
        check(lib().gtgpu_find_dev(self._h, n, d_chr, d_start, d_end, min_overlap, n_files, d_file_offsets, d_out_ids,
                                   ids_capacity, d_out_offsets, d_out_file_tok, d_out_total))


def marshal_compact(chr, start, end, file_offsets, width16_out=None, threads=0):
    """gtgpu_marshal_compact: (run_offsets, run_chr, width16, wide_index, wide_end) for gtgpu_tokenize_files_compact."""
    chr, start, end = _arr(chr, np.uint32), _arr(start, np.uint32), _arr(end, np.uint32)
    fo = _arr(file_offsets, np.uint64)
    n = len(chr)
    w16 = width16_out if width16_out is not None else np.empty(n, dtype=np.uint16)
    run_cap, wide_cap = 64 * (len(fo) - 1) + 1024, 1024
    for _ in range(2):
        ro, rc = np.empty(run_cap + 1, dtype=np.uint64), np.empty(run_cap, dtype=np.uint32)
        wi, we = np.empty(wide_cap, dtype=np.uint64), np.empty(wide_cap, dtype=np.uint32)
        n_runs, n_wide = C.c_uint64(0), C.c_uint64(0)
        st = lib().gtgpu_marshal_compact(n, _p(chr), _p(start), _p(end), len(fo) - 1, _p(fo), threads, _p(w16), run_cap, _p(ro),
                                         _p(rc), C.byref(n_runs), wide_cap, _p(wi), _p(we), C.byref(n_wide))
        if st == 4:  # GTGPU_ERR_CAPACITY: the needed counts came back
            run_cap, wide_cap = max(n_runs.value, 1), max(n_wide.value, 1)
            continue
        check(st)
        return ro[:n_runs.value + 1], rc[:n_runs.value], w16, wi[:n_wide.value], we[:n_wide.value]
    raise GtarsGpuError(4, "marshal_compact: capacity retry failed")


def marshal_packed(chr, start, end, file_offsets, width_bits=0, packed_out=None, anchors_out=None, threads=0):
    """gtgpu_marshal_packed: (run_offsets, run_chr, width_bits, packed, anchors, exc_index, exc_start, exc_end) for
    gtgpu_tokenize_files_packed."""
    chr, start, end = _arr(chr, np.uint32), _arr(start, np.uint32), _arr(end, np.uint32)
    fo = _arr(file_offsets, np.uint64)
    n = len(chr)
    pk = packed_out if packed_out is not None else np.empty(n, dtype=np.uint32)
    an = anchors_out if anchors_out is not None else np.empty((n + 31) // 32, dtype=np.uint32)
    run_cap, exc_cap = 64 * (len(fo) - 1) + 1024, 32 * (64 * (len(fo) - 1) + 1024)
    for _ in range(2):
        ro, rc = np.empty(run_cap + 1, dtype=np.uint64), np.empty(run_cap, dtype=np.uint32)
        xi, xs, xe = np.empty(exc_cap, dtype=np.uint64), np.empty(exc_cap, dtype=np.uint32), np.empty(exc_cap, dtype=np.uint32)
        n_runs, n_exc, wb = C.c_uint64(0), C.c_uint64(0), C.c_uint32(0)
        st = lib().gtgpu_marshal_packed(n, _p(chr), _p(start), _p(end), len(fo) - 1, _p(fo), threads, width_bits, _p(pk), _p(an),
                                        run_cap, _p(ro), _p(rc), C.byref(n_runs), exc_cap, _p(xi), _p(xs), _p(xe), C.byref(n_exc),
                                        C.byref(wb))
        if st == 4:  # GTGPU_ERR_CAPACITY: the needed counts came back
            run_cap, exc_cap = max(n_runs.value, 1), max(n_exc.value, 1)
            continue
        check(st)
        return (ro[:n_runs.value + 1], rc[:n_runs.value], wb.value, pk, an, xi[:n_exc.value], xs[:n_exc.value], xe[:n_exc.value])
    raise GtarsGpuError(4, "marshal_packed: capacity retry failed")


def gzip_members(gz: bytes) -> np.ndarray:
    """gtgpu_gzip_members: offsets (n_members + 1) of the gzip members of `gz` (BGZF blocks split, else one member)."""
    n = C.c_uint64(0)
    st = lib().gtgpu_gzip_members(gz, len(gz), 0, None, C.byref(n))
    if st not in (0, 4):
        check(st)
    offs = np.zeros(n.value + 1, dtype=np.uint64)
    check(lib().gtgpu_gzip_members(gz, len(gz), len(offs), _p(offs), C.byref(n)))
    return offs


def gunzip(ctx: "Context", gz: bytes, member_offsets=None):
    """gtgpu_gunzip: (text bytes, member text offsets); member_offsets default = gzip_members(gz)."""
    mo = _arr(member_offsets if member_offsets is not None else gzip_members(gz), np.uint64)
    out_off = np.zeros(len(mo), dtype=np.uint64)
    h = C.c_void_p()
    check(lib().gtgpu_gunzip(ctx._h, len(mo) - 1, gz, _p(mo), C.byref(h), _p(out_off)))
    return _take(h, dtype=np.uint8).tobytes(), out_off


def _text_ptr(text):
    """bytes, or a uint8 numpy array (a multi-GB text need not be copied into a bytes object)"""
    return _p(text) if isinstance(text, np.ndarray) else text


def _text_len(text):
    return text.nbytes if isinstance(text, np.ndarray) else len(text)


def _names_blob(chrom_names):
    blob = b"".join(n.encode() for n in chrom_names)
    offs = np.zeros(len(chrom_names) + 1, dtype=np.uint32)
    offs[1:] = np.cumsum([len(n.encode()) for n in chrom_names])
    return blob, offs


def comm_unique_id() -> bytes:
    buf = (C.c_uint8 * 128)()
    check(lib().gtgpu_comm_unique_id(buf))
    return bytes(buf)


def comm_init(ctx: Context, world: int, rank: int, uid: bytes):
    buf = (C.c_uint8 * 128).from_buffer_copy(uid)
    check(lib().gtgpu_comm_init(ctx._h, world, rank, buf))


class Igd:
    """gtgpu_igd: pooled start-sorted database records on the device (gtars-igd/src/igd.rs)."""

    def __init__(self, ctx: Context, file_offsets, n_chroms, chr, start, end):
        self.ctx = ctx
        fo = _arr(file_offsets, np.uint64)
        chr, start, end = _arr(chr, np.uint32), _arr(start, np.uint32), _arr(end, np.uint32)
        self.n_files = len(fo) - 1
        self._h = C.c_void_p()
        check(lib().gtgpu_igd_build(ctx._h, self.n_files, _p(fo), n_chroms, _p(chr), _p(start), _p(end), C.byref(self._h)))

    @classmethod
    def _from_bed(cls, ctx, n_files, call):
        obj = cls.__new__(cls)
        obj.ctx, obj.n_files, obj._h = ctx, n_files, C.c_void_p()
        nc, hn, hno = C.c_uint32(0), C.c_void_p(), C.c_void_p()
        check(call(C.byref(nc), C.byref(hn), C.byref(hno), C.byref(obj._h)))
        names = _take(hn, dtype=np.uint8).tobytes()
        no = _take(hno, dtype=np.uint64)
        return obj, [names[int(a):int(b)].decode() for a, b in zip(no[:-1], no[1:])]

    @classmethod
    def from_bed_text(cls, ctx: Context, text, file_offsets):
        """gtgpu_igd_build_bed: file f = text[file_offsets[f]:file_offsets[f + 1]], parsed on the device.  Returns (igd,
        chromosome names in id order).  `text` may be a uint8 numpy array (a multi-GB text is not copied)."""
        fo = _arr(file_offsets, np.uint64)
        return cls._from_bed(ctx, len(fo) - 1, lambda *outs: lib().gtgpu_igd_build_bed(ctx._h, len(fo) - 1, _text_ptr(text), _p(fo), *outs))

    @classmethod
    def from_bed_gz(cls, ctx: Context, gz, file_members, member_offsets):
        """gtgpu_igd_build_bed_gz: file f = gzip members [file_members[f], file_members[f + 1]) of `gz` (member_offsets as
        gzip_members returns them), inflated and parsed on the device.  Returns (igd, chromosome names in id order)."""
        fm, mo = _arr(file_members, np.uint64), _arr(member_offsets, np.uint64)
        return cls._from_bed(ctx, len(fm) - 1, lambda *outs: lib().gtgpu_igd_build_bed_gz(ctx._h, len(fm) - 1, _p(fm), len(mo) - 1,
                                                                                          _text_ptr(gz), _p(mo), *outs))

    def close(self):
        if getattr(self, "_h", None) and getattr(self.ctx, "_h", None):
            lib().gtgpu_igd_free(self._h)
        self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def info(self) -> dict:
        a = (C.c_uint64 * 4)()
        check(lib().gtgpu_igd_info(self._h, a))
        return dict(n_files=a[0], n_records=a[1], device_bytes=a[2], lut_shift=a[3])

    def _count(self, fn, set_offsets, chr, start, end, min_overlap):
        so = _arr(set_offsets, np.uint64)
        chr, start, end = _arr(chr, np.uint32), _arr(start, np.uint32), _arr(end, np.uint32)
        out = np.zeros((len(so) - 1, self.n_files), dtype=np.uint64)
        check(fn(self._h, len(so) - 1, _p(so), _p(chr), _p(start), _p(end), min_overlap, _p(out)))
        return out

    def count_set_overlaps(self, set_offsets, chr, start, end, min_overlap=1):
        return self._count(lib().gtgpu_igd_count_set_overlaps, set_offsets, chr, start, end, min_overlap)

    def count_region_hits(self, set_offsets, chr, start, end, min_overlap=1):
        return self._count(lib().gtgpu_igd_count_region_hits, set_offsets, chr, start, end, min_overlap)

    def save_bytes(self, chrom_names):
        """gtgpu_igd_serialize: (the .igd file's bytes as uint8, every file's region count, every file's width sum), the
        database's chromosome i named chrom_names[i]."""
        blob, offs = _names_blob(chrom_names)
        regions = np.zeros(self.n_files, dtype=np.uint64)
        widths = np.zeros(self.n_files, dtype=np.uint64)
        h = C.c_void_p()
        check(lib().gtgpu_igd_serialize(self._h, len(chrom_names), blob, _p(offs), C.byref(h), _p(regions), _p(widths)))
        return _take(h, dtype=np.uint8), regions, widths

    def _count_bed(self, n_sets, chrom_names, call):
        blob, offs = _names_blob(chrom_names)
        out = np.zeros((n_sets, self.n_files), dtype=np.uint64)
        regions = np.zeros(n_sets, dtype=np.uint64)
        check(call(len(chrom_names), blob, _p(offs), _p(out), _p(regions)))
        return out, regions

    def count_bed_text(self, binary, text, file_offsets, chrom_names, min_overlap=1):
        """gtgpu_igd_count_bed: count_region_hits (binary) / count_set_overlaps of query set s = text[file_offsets[s]:file_offsets[s
        + 1]], parsed on the device; chrom_names[i] is the database's chromosome i.  Returns (uint64 [n_sets, n_files], the
        sets' region lines).  `text` may be a uint8 numpy array."""
        fo = _arr(file_offsets, np.uint64)
        n = len(fo) - 1
        return self._count_bed(n, chrom_names, lambda nn, blob, offs, out, reg: lib().gtgpu_igd_count_bed(
            self._h, 1 if binary else 0, n, _text_ptr(text), _p(fo), nn, blob, offs, min_overlap, out, reg))

    def count_bed_gz(self, binary, gz, file_members, member_offsets, chrom_names, min_overlap=1):
        """gtgpu_igd_count_bed_gz: query set s = gzip members [file_members[s], file_members[s + 1]) of `gz`, inflated and parsed on
        the device.  Returns (matrix, the sets' region lines) as count_bed_text does."""
        fm, mo = _arr(file_members, np.uint64), _arr(member_offsets, np.uint64)
        n = len(fm) - 1
        return self._count_bed(n, chrom_names, lambda nn, blob, offs, out, reg: lib().gtgpu_igd_count_bed_gz(
            self._h, 1 if binary else 0, n, _p(fm), len(mo) - 1, _text_ptr(gz), _p(mo), nn, blob, offs, min_overlap, out, reg))

    def count_sharded(self, binary, n_files_global, set_offsets, chr, start, end, min_overlap=1, out=None):
        """`out` (optional): a caller-owned uint64 [n_sets, n_files_global] array, e.g. pinned memory from pinned_empty."""
        so = _arr(set_offsets, np.uint64)
        chr, start, end = _arr(chr, np.uint32), _arr(start, np.uint32), _arr(end, np.uint32)
        if out is None:
            out = np.zeros((len(so) - 1, n_files_global), dtype=np.uint64)
        assert out.dtype == np.uint64 and out.shape == (len(so) - 1, n_files_global) and out.flags.c_contiguous
        check(lib().gtgpu_igd_count_sharded(self.ctx._h, self._h, 1 if binary else 0, n_files_global, len(so) - 1, _p(so),
                                            _p(chr), _p(start), _p(end), min_overlap, _p(out)))
        return out
