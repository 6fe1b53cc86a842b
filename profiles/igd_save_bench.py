"""Wall time of creating an .igd database from BED files: api.Igd.from_bed_files(paths).save(p, names) (parse and file written on
the device) against api.write_igd_file([RegionSet(p) ...], names, p) (host parser, host tile sort), files in the page cache;
plus gtgpu_igd_serialize alone (ffi.Igd.save_bytes) on the same database.

    python profiles/igd_save_bench.py [--sets 2000] [--per-set 20000] [--reps 3] [--out profiles/igd_save_bench.jsonl]

Workload: the seeded database of igd_bed_bench.py (--sets plain BED files of --per-set regions each).  Every arm is the best of
--reps runs after one warm-up of the device arms; the .igd and .tsv bytes of the two writers are compared.  One JSON line per
measurement, with the card's name and power limit read in the same run.  Files go to a temporary directory removed at the end.
"""
from __future__ import annotations

import argparse
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time
from multiprocessing import Pool

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "profiles"))

from igd_bed_bench import write_set  # noqa: E402
from score_text_bench import cache, timed  # noqa: E402


def read(p):
    with open(p, "rb") as f:
        return f.read()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sets", type=int, default=2000)
    ap.add_argument("--per-set", type=int, default=20_000)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "igd_save_bench.jsonl"))
    args = ap.parse_args()
    gpu, power = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                                text=True, check=True).stdout.splitlines()[0].split(", ")
    tmp = tempfile.mkdtemp(prefix="igd_save_")
    out = open(args.out, "a")

    def emit(**kv):
        kv.update(gpu=gpu, power_limit=power, sets=args.sets, per_set=args.per_set)
        print(json.dumps(kv), flush=True)
        out.write(json.dumps(kv) + "\n")
        out.flush()

    try:
        import numpy as np
        from gtars_b200 import api, ffi
        api.device(0)
        paths = [os.path.join(tmp, f"set{i:05d}.bed") for i in range(args.sets)]
        with Pool(max(1, min(32, os.cpu_count() or 1))) as pool:
            pool.map(write_set, [(p, 100 + i, args.per_set) for i, p in enumerate(paths)], chunksize=16)
        for p in paths:
            os.remove(p + ".gz")
        cache(paths)
        names = [os.path.basename(p) for p in paths]
        dev_p, host_p = os.path.join(tmp, "dev.igd"), os.path.join(tmp, "host.igd")
        api.Igd.from_bed_files(paths[:8]).save(dev_p, names[:8])  # warm-up: modules, allocator
        td, _ = timed(lambda: api.Igd.from_bed_files(paths).save(dev_p, names), reps=args.reps)
        emit(workload="igd_create", arm="device", wall_s=td, igd_bytes=os.path.getsize(dev_p))
        th, _ = timed(lambda: api.write_igd_file([api.RegionSet(p) for p in paths], names, host_p), reps=args.reps)
        emit(workload="igd_create", arm="host", wall_s=th,
             igd_equal=read(dev_p) == read(host_p), tsv_equal=read(dev_p[:-4] + ".tsv") == read(host_p[:-4] + ".tsv"))

        texts = [read(p) for p in paths]
        fo = np.cumsum([0] + [len(t) for t in texts]).astype(np.uint64)
        ctx = ffi.Context(0)
        g, chroms = ffi.Igd.from_bed_text(ctx, np.frombuffer(b"".join(texts), dtype=np.uint8), fo)
        g.save_bytes(chroms)  # warm-up
        ts, (b, _, _) = timed(lambda: g.save_bytes(chroms), reps=args.reps)
        emit(workload="gtgpu_igd_serialize", wall_s=ts, n_records=g.info()["n_records"], igd_bytes=int(b.nbytes),
             equal=b.tobytes() == read(dev_p))
        g.close()
        ctx.close()
    finally:
        out.close()
        shutil.rmtree(tmp, ignore_errors=True)


if __name__ == "__main__":
    main()
