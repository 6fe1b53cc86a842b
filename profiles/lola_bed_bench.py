"""Wall time of run_lola's contingency tables with the user sets and the universe given as BED files:
api.lola_contingency_from_bed_files (the files' text parsed on the device, one count pass) against
api.lola_contingency(igd, [RegionSet(p) ...], RegionSet(universe)) (host parser, host name map, then the same count kernel).

    python profiles/lola_bed_bench.py [--db-sets 10000] [--db-per-set 20000] [--user-sets 1000] [--per-user 10000]
                                      [--universe 1000000] [--out profiles/lola_bed_bench.jsonl]

Workload (C4's shape at the defaults): a seeded database of --db-sets BED files of --db-per-set regions, loaded once with
api.Igd.from_bed_files; --user-sets user sets of --per-user regions sampled from a --universe-region universe, and the
universe itself, written as plain .bed and as one-member .bed.gz files and read once to warm the page cache.  Both arms on
both forms: best of 3 after a warm-up, with a flag saying whether the two int64 tables are equal.  One JSON line per
measurement, each with the card's name and power limit read in the same run.  Files go to a temporary directory that is
removed at the end.
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


def bed_bytes(c, s, e):
    """BED lines "name\\tstart\\tend\\n" of the arrays, built with numpy (coordinates zero-padded to 10 digits)"""
    from gtars_b200 import synth
    names = [n.encode() for n in synth.CHROM_NAMES[:N_CHROMS]]
    tab = np.zeros((len(names), 8), dtype=np.uint8)
    for i, n in enumerate(names):
        tab[i, :len(n)] = list(n)
    nl = np.array([len(n) for n in names], dtype=np.int64)[c]
    off = np.zeros(len(c) + 1, dtype=np.int64)
    np.cumsum(nl + 23, out=off[1:])
    out = np.empty(int(off[-1]), dtype=np.uint8)
    a = off[:-1]
    for j in range(int(nl.max())):
        m = nl > j
        out[a[m] + j] = tab[c[m], j]
    p = a + nl
    out[p], out[p + 11], out[p + 22] = 9, 9, 10
    for col, v in ((p + 1, s), (p + 12, e)):
        v = np.asarray(v).astype(np.uint64)
        for j in range(9, -1, -1):
            out[col + j] = (v % 10).astype(np.uint8) + 48
            v //= 10
    return out.tobytes()


def records(n, seed, width=(100, 10_000)):
    rng = np.random.default_rng(seed)
    c = rng.integers(0, N_CHROMS, n).astype(np.int64)
    s = rng.integers(0, 2**28, n).astype(np.uint32)
    return c, s, (s + rng.integers(width[0], width[1], n)).astype(np.uint32)


def write_db_set(args):
    path, seed, per = args
    with open(path, "wb") as f:
        f.write(bed_bytes(*records(per, seed)))


_UNIVERSE = None  # (chr, start, end) of the universe, set in every writer process


def _init(universe):
    global _UNIVERSE
    _UNIVERSE = universe


def write_query(args):
    """one user set (rows of the universe) or the universe itself, plain and one-member gzip"""
    path, rows = args
    c, s, e = _UNIVERSE
    text = bed_bytes(c[rows], s[rows], e[rows])
    with open(path, "wb") as f:
        f.write(text)
    with open(path + ".gz", "wb") as f:
        f.write(gzip.compress(text, compresslevel=6, mtime=0))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--db-sets", type=int, default=10_000)
    ap.add_argument("--db-per-set", type=int, default=20_000)
    ap.add_argument("--user-sets", type=int, default=1000)
    ap.add_argument("--per-user", type=int, default=10_000)
    ap.add_argument("--universe", type=int, default=1_000_000)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "lola_bed_bench.jsonl"))
    args = ap.parse_args()
    gpu, power = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                                text=True, check=True).stdout.splitlines()[0].split(", ")
    tmp = tempfile.mkdtemp(prefix="lola_bed_")
    out = open(args.out, "a")
    shape = dict(db_sets=args.db_sets, db_per_set=args.db_per_set, user_sets=args.user_sets, per_user=args.per_user,
                 universe=args.universe)

    def emit(**kv):
        kv.update(shape)
        kv.update(gpu=gpu, power_limit=power)
        print(json.dumps(kv), flush=True)
        out.write(json.dumps(kv) + "\n")
        out.flush()

    try:
        from gtars_b200 import api
        api.device(0)
        procs = max(1, min(32, os.cpu_count() or 1))
        t = time.perf_counter()
        db_paths = [os.path.join(tmp, f"db{i:05d}.bed") for i in range(args.db_sets)]
        with Pool(procs) as pool:
            pool.map(write_db_set, [(p, 100 + i, args.db_per_set) for i, p in enumerate(db_paths)], chunksize=16)
        universe = records(args.universe, 7, width=(100, 5000))
        rng = np.random.default_rng(8)
        user_paths = [os.path.join(tmp, f"user{i:04d}.bed") for i in range(args.user_sets)]
        universe_path = os.path.join(tmp, "universe.bed")
        jobs = [(p, np.sort(rng.choice(args.universe, args.per_user, replace=False))) for p in user_paths]
        jobs.append((universe_path, np.arange(args.universe)))
        with Pool(procs, initializer=_init, initargs=(universe,)) as pool:
            pool.map(write_query, jobs, chunksize=8)
        emit(workload="write_files", wall_s=time.perf_counter() - t)
        cache(db_paths)
        t = time.perf_counter()
        db = api.Igd.from_bed_files(db_paths)
        emit(workload="igd_from_bed_files", wall_s=time.perf_counter() - t, n_records=db.info()["n_records"])
        for fmt, ups, up in (("plain", user_paths, universe_path),
                             ("gzip", [p + ".gz" for p in user_paths], universe_path + ".gz")):
            cache(ups + [up])
            size = sum(os.path.getsize(p) for p in ups + [up])
            api.lola_contingency_from_bed_files(db, ups, up)                     # warm-up
            td, dev = timed(lambda: api.lola_contingency_from_bed_files(db, ups, up), reps=args.reps)
            emit(workload="lola_contingency", format=fmt, file_bytes=size, arm="device_parse", wall_s=td,
                 a_sum=int(dev[:, :, 0].sum()))
            host_arm = lambda: api.lola_contingency(db, [api.RegionSet(p) for p in ups], api.RegionSet(up))  # noqa: E731
            host_arm()                                                           # warm-up
            th, host = timed(host_arm, reps=args.reps)
            emit(workload="lola_contingency", format=fmt, file_bytes=size, arm="host_parse", wall_s=th,
                 equal=bool(np.array_equal(host, dev)), speedup=th / td)
            del dev, host
        # one member, one warp: the device inflater's time for the universe's single gzip member alone
        from gtars_b200 import ffi
        ctx = ffi.Context(0)
        gz = open(universe_path + ".gz", "rb").read()
        ffi.gunzip(ctx, gz)
        tg, _ = timed(lambda: ffi.gunzip(ctx, gz), reps=args.reps)
        emit(workload="gunzip_universe", gz_bytes=len(gz), wall_s=tg)
        ctx.close()
    finally:
        out.close()
        shutil.rmtree(tmp, ignore_errors=True)


if __name__ == "__main__":
    main()
