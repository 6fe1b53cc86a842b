"""Wall time of resolving a batch of BED query files against a MultiChromOverlapper two ways that give the same answer: the host
path (RegionSet(p) parsed and sorted on one host core, then the existing count_overlaps / find_overlaps / subset_by per file)
and the one-pass device path (count_overlaps_bed_files / find_overlaps_bed_files / subset_by_bed_files: every file parsed,
sorted and resolved on the device); files already in the page cache.

    python profiles/overlaps_bed_files_bench.py [--files 1000] [--regions 100000] [--source 1000000] [--reps 3] [--out PATH]

Workload: the corpus of profiles/tokenize_bed_files_bench.py (C2's shape, seeded gtars_b200.synth): --files query files of
--regions regions, plain .bed and one-member .bed.gz, against an AIList overlapper over the --source-region universe file.  The
two answers are asserted equal for every operation and form (subset_by: every file's size and every region of every 50th
file).  One JSON line per measurement, each with the card's name and power
limit read in the same run.  Files go to a temporary directory that is removed at the end.
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

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "profiles"))

from score_text_bench import cache, timed  # noqa: E402
from tokenize_bed_files_bench import write_corpus  # noqa: E402


def flat_hits(per_query):
    """per-query hit lists -> (per-query counts, concatenated hits)"""
    lens = np.fromiter((len(h) for h in per_query), dtype=np.int64, count=len(per_query))
    vals = np.fromiter((v for h in per_query for v in h), dtype=np.uint32, count=int(lens.sum()))
    return lens, vals


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--files", type=int, default=1000)
    ap.add_argument("--regions", type=int, default=100_000, help="regions per file")
    ap.add_argument("--source", type=int, default=1_000_000, help="regions of the overlapper's source")
    ap.add_argument("--reps", type=int, default=3, help="timed repetitions of the device arm (best is reported); the host arm runs once")
    ap.add_argument("--out", help="also append the JSON lines to this file")
    args = ap.parse_args()
    tmp = tempfile.mkdtemp(prefix="overlaps_bed_files_")
    out = open(args.out, "a") if args.out else None

    gpu, power = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                                text=True, check=True).stdout.splitlines()[0].split(", ")

    def emit(**kv):
        kv.update(gpu=gpu, power_limit=power)
        print(json.dumps(kv), flush=True)
        if out:
            out.write(json.dumps(kv) + "\n")
            out.flush()

    try:
        t = time.perf_counter()
        spath, paths = write_corpus(tmp, args.files, args.regions, args.source)
        forms = {"plain": paths, "gzip": [p + ".gz" for p in paths]}
        emit(workload="write_files", files=args.files, per_file=args.regions, source=args.source, wall_s=time.perf_counter() - t,
             file_bytes={k: sum(os.path.getsize(p) for p in v) for k, v in forms.items()})
        from gtars_b200 import api
        api.device(0)
        mco = api.MultiChromOverlapper(api.RegionSet(spath), api.AILIST)
        for form, ps in forms.items():
            cache(ps)
            size = sum(os.path.getsize(p) for p in ps)
            mco.count_overlaps_bed_files(ps[:2])                               # warm-up: modules, allocator, pinned blocks
            # (host arm, device arm, equality of their answers; not timed)
            ops = {
                "count": (lambda: [mco.count_overlaps(api.RegionSet(p)) for p in ps],
                          lambda: mco.count_overlaps_bed_files(ps),
                          lambda h, d: all(np.array_equal(np.asarray(a, dtype=np.uint32), b) for a, b in zip(h, d))),
                "find": (lambda: [mco.find_overlaps(api.RegionSet(p)) for p in ps],
                         lambda: mco.find_overlaps_bed_files(ps),
                         lambda h, d: all(np.array_equal(flat_hits(a)[0], np.diff(o)) and np.array_equal(flat_hits(a)[1], v)
                                          for a, (o, v) in zip(h, d))),
                # every file's size, and every region of every 50th file (a region is read through ctypes one at a time)
                "subset_by": (lambda: [mco.subset_by(api.RegionSet(p)) for p in ps],
                              lambda: mco.subset_by_bed_files(ps),
                              lambda h, d: [len(a) for a in h] == [len(b) for b in d] and all(list(h[f]) == list(d[f])
                                                                                             for f in range(0, len(h), 50))),
            }
            for op, (host, device, same) in ops.items():
                t = time.perf_counter()
                want = host()
                host_s = time.perf_counter() - t
                dev_s, got = timed(device, reps=args.reps)
                assert len(got) == len(want) and same(want, got), (form, op)
                base = dict(workload="overlaps_bed_files", op=op, files=args.files, per_file=args.regions, source=args.source,
                            format=form, file_bytes=size, equal=True)
                emit(**base, arm="host_regionset_per_file", wall_s=host_s)
                emit(**base, arm="device_bed_files", wall_s=dev_s, speedup=host_s / dev_s)
                del want, got
    finally:
        if out:
            out.close()
        shutil.rmtree(tmp, ignore_errors=True)


if __name__ == "__main__":
    main()
