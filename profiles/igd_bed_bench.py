"""Wall time of loading an IGD database from its BED files: api.Igd.from_bed_files(paths) (text parsed on the device) against
api.Igd([RegionSet(p) for p in paths]) (host parser), files already in the page cache; plus gtgpu_igd_build_bed / _gz on the
same files and gtgpu_igd_build on C4-shaped arrays for two builds of the library timed alternately.

    python profiles/igd_bed_bench.py [--sets 10000] [--per-set 20000] [--out profiles/igd_bed_bench.jsonl] [--lib PATH ...]

Workloads: a seeded database of --sets BED files of --per-set regions each (C4's shape at the defaults: 1e4 x 2e4), written
as plain .bed and as one-member .bed.gz files; both loaders on both forms, with the count matrices of one query batch (64
sets x 2 000 regions) compared between them.  Then, through each library given with --lib (default: the in-tree one), in
alternating child processes: gtgpu_igd_build_bed and _gz (ffi.Igd.from_bed_text / from_bed_gz) on the same files, and
gtgpu_igd_build (ffi.Igd) on 1e4 x 2e4 records.  One JSON line per measurement, each with the card's
name and power limit read in the same run.  Files go to a temporary directory that is removed at the end.
"""
from __future__ import annotations

import argparse
import gzip
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time
from multiprocessing import Pool

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "profiles"))

from score_text_bench import cache, timed  # noqa: E402

N_CHROMS = 25


def records(n, seed):
    rng = np.random.default_rng(seed)
    c = rng.integers(0, N_CHROMS, n).astype(np.int64)
    s = rng.integers(0, 2**28, n).astype(np.uint32)
    return c, s, (s + rng.integers(100, 10_000, n)).astype(np.uint32)


def bed_lines(c, s, e):
    from gtars_b200 import synth
    return "".join(f"{synth.CHROM_NAMES[x]}\t{y}\t{z}\n" for x, y, z in zip(c.tolist(), s.tolist(), e.tolist())).encode()


def write_set(args):
    path, seed, per = args
    text = bed_lines(*records(per, seed))
    with open(path, "wb") as f:
        f.write(text)
    with open(path + ".gz", "wb") as f:
        f.write(gzip.compress(text, compresslevel=6, mtime=0))


def child_ffi():
    """the ffi of the library named by GTGPU_LIB (set by the parent)"""
    import ctypes
    from gtars_b200 import ffi
    exported = ctypes.CDLL(ffi.LIB_PATH)
    for name in [n for n in ffi.SIGNATURES if not hasattr(exported, n)]:  # an older build lacks entry points added since
        del ffi.SIGNATURES[name]
    return ffi


def load_child(tmp, n_sets, reps):
    """Child process: best wall time of gtgpu_igd_build_bed (the plain files back to back) and gtgpu_igd_build_bed_gz (one
    member per file) over the files in tmp, with a checksum of one query batch's counts."""
    from gtars_b200 import synth
    ffi = child_ffi()
    paths = [os.path.join(tmp, f"set{i:05d}.bed") for i in range(n_sets)]
    texts = [open(p, "rb").read() for p in paths]
    gzs = [open(p + ".gz", "rb").read() for p in paths]
    text, gz = np.frombuffer(b"".join(texts), dtype=np.uint8), np.frombuffer(b"".join(gzs), dtype=np.uint8)
    fo = np.cumsum([0] + [len(t) for t in texts]).astype(np.uint64)
    mo = np.cumsum([0] + [len(g) for g in gzs]).astype(np.uint64)
    qc, qs, qe = records(64 * 2000, 7)
    so = np.arange(0, 64 * 2000 + 1, 2000, dtype=np.uint64)
    ctx = ffi.Context(0)
    res = {}
    for fmt, call in (("plain", lambda: ffi.Igd.from_bed_text(ctx, text, fo)),
                      ("gzip", lambda: ffi.Igd.from_bed_gz(ctx, gz, np.arange(n_sets + 1, dtype=np.uint64), mo))):
        call()[0].close()                                                # warm-up: modules, allocator
        best = None
        for _ in range(reps):
            t = time.perf_counter()
            g, names = call()
            dt = time.perf_counter() - t
            best = dt if best is None else min(best, dt)
            if _ < reps - 1:
                g.close()
        idx = {n: i for i, n in enumerate(names)}
        remap = np.array([idx.get(n, 0xFFFFFFFF) for n in synth.CHROM_NAMES[:N_CHROMS]], dtype=np.uint32)
        cnt = g.count_set_overlaps(so, remap[qc], qs, qe)
        res[fmt] = dict(wall_s=best, n_records=g.info()["n_records"], names=len(names), counts_sum=int(cnt.sum()))
        g.close()
    ctx.close()
    print(json.dumps(res))


def build_child(n_sets, per, reps):
    """Child process: best wall time of gtgpu_igd_build over C4-shaped arrays."""
    ffi = child_ffi()
    c, s, e = records(n_sets * per, 1)
    fo = np.arange(n_sets + 1, dtype=np.uint64) * np.uint64(per)
    c = c.astype(np.uint32)
    ctx = ffi.Context(0)
    ffi.Igd(ctx, fo, N_CHROMS, c, s, e).close()                          # warm-up: modules, allocator
    t, g = timed(lambda: ffi.Igd(ctx, fo, N_CHROMS, c, s, e), reps=reps)
    so = np.array([0, 1000], dtype=np.uint64)
    cnt = g.count_region_hits(so, c[:1000], s[:1000], e[:1000])
    print(json.dumps(dict(wall_s=t, n_records=g.info()["n_records"], counts_sum=int(cnt.sum()))))
    g.close()
    ctx.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sets", type=int, default=10_000)
    ap.add_argument("--per-set", type=int, default=20_000)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "igd_bed_bench.jsonl"))
    ap.add_argument("--lib", action="append", help="libgtars_gpu.so to time gtgpu_igd_build with (repeatable; default: in-tree)")
    ap.add_argument("--rounds", type=int, default=3, help="alternating rounds of the build comparison")
    ap.add_argument("--only-build", action="store_true", help="run the build comparison only")
    ap.add_argument("--build-child", action="store_true", help=argparse.SUPPRESS)
    ap.add_argument("--load-child", help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.build_child:
        build_child(10_000, 20_000, 3)
        return
    if args.load_child:
        load_child(args.load_child, args.sets, 3)
        return
    gpu, power = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                                text=True, check=True).stdout.splitlines()[0].split(", ")
    tmp = tempfile.mkdtemp(prefix="igd_bed_")
    out = open(args.out, "a")

    def emit(**kv):
        kv.update(gpu=gpu, power_limit=power)
        print(json.dumps(kv), flush=True)
        out.write(json.dumps(kv) + "\n")
        out.flush()

    try:
        if not args.only_build:
            from gtars_b200 import api, synth
            api.device(0)
            paths = [os.path.join(tmp, f"set{i:05d}.bed") for i in range(args.sets)]
            t = time.perf_counter()
            with Pool(max(1, min(32, os.cpu_count() or 1))) as pool:
                pool.map(write_set, [(p, 100 + i, args.per_set) for i, p in enumerate(paths)], chunksize=16)
            emit(workload="write_files", sets=args.sets, per_set=args.per_set, wall_s=time.perf_counter() - t)
            qc, qs, qe = records(64 * 2000, 7)
            queries = [[(synth.CHROM_NAMES[x], y, z) for x, y, z in zip(qc[k:k + 2000].tolist(), qs[k:k + 2000].tolist(), qe[k:k + 2000].tolist())]
                       for k in range(0, len(qc), 2000)]
            for fmt, ps in (("plain", paths), ("gzip", [p + ".gz" for p in paths])):
                cache(ps)
                size = sum(os.path.getsize(p) for p in ps)
                td, dev = timed(lambda: api.Igd.from_bed_files(ps))
                want = dev._count(queries, 1, False)
                emit(workload="igd_from_bed_files", sets=args.sets, per_set=args.per_set, format=fmt, file_bytes=size, arm="device_parse",
                     wall_s=td, n_records=dev.info()["n_records"])
                del dev
                th, host = timed(lambda: api.Igd([api.RegionSet(p) for p in ps]))
                emit(workload="igd_from_bed_files", sets=args.sets, per_set=args.per_set, format=fmt, file_bytes=size, arm="host_parse",
                     wall_s=th, equal=bool(np.array_equal(host._count(queries, 1, False), want)))
                del host
        libs = args.lib or [os.path.join(ROOT, "gtars_b200", "libgtars_gpu.so")]
        if not args.only_build:
            for r in range(args.rounds):
                for lib in libs:
                    env = dict(os.environ, GTGPU_LIB=os.path.abspath(lib))
                    res = subprocess.run([sys.executable, os.path.abspath(__file__), "--load-child", tmp, "--sets", str(args.sets)],
                                         env=env, capture_output=True, text=True, check=True)
                    for fmt, kv in json.loads(res.stdout.strip().splitlines()[-1]).items():
                        emit(workload="gtgpu_igd_build_bed", sets=args.sets, per_set=args.per_set, format=fmt, lib=lib, round=r, **kv)
        for r in range(args.rounds):
            for lib in libs:
                env = dict(os.environ, GTGPU_LIB=os.path.abspath(lib))
                res = subprocess.run([sys.executable, os.path.abspath(__file__), "--build-child"], env=env, capture_output=True, text=True,
                                     check=True)
                emit(workload="gtgpu_igd_build_c4", sets=10_000, per_set=20_000, lib=lib, round=r,
                     **json.loads(res.stdout.strip().splitlines()[-1]))
    finally:
        out.close()
        shutil.rmtree(tmp, ignore_errors=True)


if __name__ == "__main__":
    main()
