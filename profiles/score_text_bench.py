"""Wall time of region_scoring_from_fragments / barcode_scoring_from_fragments with the host parse vs device_parse=True,
files already in the page cache, plus a device-side split of the text path.

    python profiles/score_text_bench.py [--scale 1.0] [--out profiles/score_text_bench.jsonl]

Workloads (at --scale 1): the README's scoring workload as files (8 x 2.5e7 fragments vs 1 M peaks, ATAC), one barcode
file of 1e8 fragments, each as plain text and as BGZF; and one plain file of 1.1e8 fragments (> 4 GiB), device only.  One
JSON line per measurement, each with the card's name and power limit read in the same run.  Files go to a temporary
directory that is removed at the end.

Device split (ffi level, same universe): `h2d_parse` = gtgpu_score_matrix_text with n_cols = 0 (the parse runs, the
find is skipped); `score` = the full call minus that; `find_kernel` / `inflate_kernel` = CUDA-event times of the fused
find and gunzip kernels (gtgpu_timing_*); `inflate_parse` = gtgpu_score_matrix_gz with n_cols = 0.  The first three are
host-clock differences around synchronised calls, the kernel times come from events.
"""
from __future__ import annotations

import argparse
import json
import os
import shutil
import struct
import subprocess
import sys
import tempfile
import time
import zlib
from multiprocessing import Pool

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def _deflate(block: bytes) -> bytes:
    co = zlib.compressobj(1, zlib.DEFLATED, -15)
    body = co.compress(block) + co.flush()
    return (b"\x1f\x8b\x08\x04" + b"\0" * 4 + b"\x00\xff" + struct.pack("<H", 6) + b"BC" + struct.pack("<HH", 2, 12 + 6 + len(body) + 8 - 1)
            + body + struct.pack("<II", zlib.crc32(block), len(block)))


def write_bgzf(path, text: np.ndarray, pool, block=65_280):
    mv = memoryview(text)
    with open(path, "wb") as f:
        for part in pool.imap(_deflate, (bytes(mv[i:i + block]) for i in range(0, len(text), block)), chunksize=64):
            f.write(part)
        f.write(_deflate(b""))


def write_fragments(path, n, seed, n_barcodes, pool=None, chunk=10_000_000):
    from gtars_b200 import synth
    with open(path, "wb") as f:
        for k, a in enumerate(range(0, n, chunk)):
            f.write(synth.fragment_text(*synth.make_fragment_arrays(min(chunk, n - a), seed * 1000 + k, n_barcodes)).tobytes())
    if pool is not None:
        text = np.fromfile(path, dtype=np.uint8)
        write_bgzf(path + ".gz", text, pool)


def cache(paths):
    for p in paths:
        with open(p, "rb") as f:
            while f.read(1 << 26):
                pass


def timed(fn, reps=1):
    best = None
    for _ in range(reps):
        t = time.perf_counter()
        out = fn()
        dt = time.perf_counter() - t
        best = dt if best is None else min(best, dt)
    return best, out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--scale", type=float, default=1.0)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "score_text_bench.jsonl"))
    ap.add_argument("--no-host", action="store_true", help="skip the host-parse arms")
    args = ap.parse_args()
    from gtars_b200 import api, ffi, synth
    gpu, power = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                                text=True, check=True).stdout.splitlines()[0].split(", ")
    tmp = tempfile.mkdtemp(prefix="score_text_")
    out = open(args.out, "a")

    def emit(**kv):
        kv.update(gpu=gpu, power_limit=power, scale=args.scale)
        print(json.dumps(kv), flush=True)
        out.write(json.dumps(kv) + "\n")
        out.flush()

    try:
        u = synth.make_universe(1_000_000)
        uc, us, ue = (u[k].numpy() for k in ("chr", "start", "end"))
        order = np.lexsort((us, np.array([synth.CHROM_NAMES[i] for i in range(len(synth.CHROM_NAMES))])[uc]))
        cons_path = os.path.join(tmp, "consensus.bed")
        with open(cons_path, "w") as f:
            f.write("".join(f"{synth.CHROM_NAMES[c]}\t{s}\t{e}\n" for c, s, e in zip(uc[order], us[order], ue[order])))
        cons = api.ConsensusSet(cons_path)
        pool = Pool(max(1, min(32, os.cpu_count() or 1)))

        # ---- region scoring: 8 files x 2.5e7 fragments ----
        n_file = int(25_000_000 * args.scale)
        files = [os.path.join(tmp, f"frag{f}.tsv") for f in range(8)]
        for f, p in enumerate(files):
            write_fragments(p, n_file, 10 + f, 100_000, pool)
        for fmt, paths in (("plain", files), ("bgzf", [p + ".gz" for p in files])):
            cache(paths)
            tb = sum(os.path.getsize(p) for p in paths)
            td, md = timed(lambda: api.region_scoring_from_fragments(paths, cons, api.SCORING_ATAC, device_parse=True), reps=2)
            emit(workload="region_scoring_8x", fragments=8 * n_file, format=fmt, file_bytes=tb, arm="device_parse", wall_s=td)
            if not args.no_host:
                th, mh = timed(lambda: api.region_scoring_from_fragments(paths, cons, api.SCORING_ATAC))
                emit(workload="region_scoring_8x", fragments=8 * n_file, format=fmt, file_bytes=tb, arm="host_parse", wall_s=th,
                     equal=bool(np.array_equal(md, mh)))
        for p in files:
            os.remove(p)
            os.remove(p + ".gz")

        # ---- barcode scoring: one file of 1e8 fragments ----
        n_bc = int(100_000_000 * args.scale)
        bpath = os.path.join(tmp, "barcodes.tsv")
        write_fragments(bpath, n_bc, 99, 1_000_000, pool)
        for fmt, p in (("plain", bpath), ("bgzf", bpath + ".gz")):
            cache([p])
            td, dd = timed(lambda: api.barcode_scoring_from_fragments(p, cons, device_parse=True))
            emit(workload="barcode_scoring", fragments=n_bc, format=fmt, file_bytes=os.path.getsize(p), arm="device_parse", wall_s=td,
                 barcodes=len(dd))
            if not args.no_host:
                th, dh = timed(lambda: api.barcode_scoring_from_fragments(p, cons))
                emit(workload="barcode_scoring", fragments=n_bc, format=fmt, file_bytes=os.path.getsize(p), arm="host_parse", wall_s=th,
                     equal=dd == dh)
            del dd
        os.remove(bpath)
        os.remove(bpath + ".gz")

        # ---- > 4 GiB of plain text, device only ----
        n_big = int(110_000_000 * args.scale)
        big = os.path.join(tmp, "big.tsv")
        write_fragments(big, n_big, 7, 1_000_000)
        cache([big])
        td, _ = timed(lambda: api.region_scoring_from_fragments([big], cons, api.SCORING_ATAC, device_parse=True))
        emit(workload="region_scoring_big", fragments=n_big, format="plain", file_bytes=os.path.getsize(big), arm="device_parse", wall_s=td)
        os.remove(big)

        # ---- device split of one 2.5e7-fragment file (ffi level, text already in host memory) ----
        offs = u["chrom_offsets"].numpy().astype(np.uint64)
        s, e, v = (u[k].numpy().view(np.uint32) for k in ("g_start", "g_end", "g_val"))
        ctx = ffi.Context(0)
        ix = ffi.Index(ctx, ffi.KIND_BITS, offs, s, e, v)
        text = synth.fragment_text(*synth.make_fragment_arrays(n_file, 10, 100_000))
        gz_path = os.path.join(tmp, "split.tsv.gz")
        write_bgzf(gz_path, text, pool)
        gz = open(gz_path, "rb").read()
        mo = ffi.gzip_members(gz)
        names, n_cols = synth.CHROM_NAMES, int(u["n"])
        ix.score_matrix_text(text, names, ffi.SCORE_ATAC, n_cols)              # warm-up
        t_parse, _ = timed(lambda: ix.score_matrix_text(text, names, ffi.SCORE_ATAC, 0), reps=3)
        ctx.timing_enable(True)
        t_full, _ = timed(lambda: ix.score_matrix_text(text, names, ffi.SCORE_ATAC, n_cols), reps=3)
        find_ms = ctx.timing_read()
        t_gz, _ = timed(lambda: ix.score_matrix_text(gz, names, ffi.SCORE_ATAC, 0, gz_member_offsets=mo), reps=3)
        inflate_ms = ctx.timing_read()
        ctx.timing_enable(False)
        emit(workload="device_split_one_file", fragments=n_file, text_bytes=int(text.nbytes), gz_bytes=len(gz),
             h2d_parse_s=t_parse, score_s=t_full - t_parse, full_text_s=t_full, inflate_parse_s=t_gz,
             find_kernel_ms=min(find_ms) if find_ms else None, inflate_kernel_ms=min(inflate_ms) if inflate_ms else None)
        ix.close()
        ctx.close()
        pool.close()
    finally:
        out.close()
        shutil.rmtree(tmp, ignore_errors=True)


if __name__ == "__main__":
    main()
