"""Wall time of tokenizing a batch of BED files three ways that give the same answer: tok.encode_batch(paths) (every file
parsed and sorted on one host core, then one device pass), [tok.encode_bed_file(p) for p in paths] (one device parse and
round trip per file) and tok.encode_bed_files(paths) (one device pass over all the files' text); files already in the page
cache.

    python profiles/tokenize_bed_files_bench.py [--files 1000] [--regions 100000] [--universe 1000000] [--reps 3] [--out PATH]

Workload: C2's shape at a reduced default size, seeded (gtars_b200.synth): --files query files of --regions regions against a
--universe-peak tokenizer, written as plain .bed and as one-member .bed.gz files, both sorted by (chromosome name, start) as
RegionSet writes them, plus the plain files with their lines shuffled ("unsorted", which the device sorts back per file).
The three answers are asserted equal for every form.  One JSON line per measurement, each with the card's name and power
limit read in the same run.  Files go to a temporary directory that is removed at the end.  --write-only writes the corpus
and stops (no device needed).
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


def bed_bytes(chr_id, start, end):
    """ "name\\tstart\\tend\\n" lines (plain decimal coordinates) for synth chromosome ids, vectorised."""
    from gtars_b200 import synth
    names = [n.encode() for n in synth.CHROM_NAMES]
    tab = np.zeros((len(names), max(len(n) for n in names)), dtype=np.uint8)
    for i, n in enumerate(names):
        tab[i, :len(n)] = list(n)
    chr_id = np.asarray(chr_id, dtype=np.int64)
    cols = [np.asarray(v, dtype=np.uint64) for v in (start, end)]
    digits = [np.maximum(1, np.floor(np.log10(np.maximum(v, 1).astype(np.float64))).astype(np.int64) + 1) for v in cols]
    nl = np.array([len(n) for n in names], dtype=np.int64)[chr_id]
    off = np.zeros(len(chr_id) + 1, dtype=np.int64)
    np.cumsum(nl + digits[0] + digits[1] + 3, out=off[1:])
    out = np.empty(int(off[-1]), dtype=np.uint8)
    a = off[:-1]
    for j in range(int(nl.max(initial=0))):
        m = nl > j
        out[a[m] + j] = tab[chr_id[m], j]
    p = a + nl
    for v, d in zip(cols, digits):
        out[p] = 9
        v = v.copy()
        for j in range(int(d.max(initial=1))):
            m = d > j
            out[(p + d - j)[m]] = (v[m] % 10).astype(np.uint8) + 48
            v //= 10
        p = p + d + 1
    out[p] = 10
    return out.tobytes()


def write_file(args):
    path, c, s, e, seed = args
    text = bed_bytes(c, s, e)
    with open(path, "wb") as f:
        f.write(text)
    with open(path + ".gz", "wb") as f:
        f.write(gzip.compress(text, compresslevel=6, mtime=0))
    perm = np.random.default_rng(seed).permutation(len(c))
    with open(path[:-4] + ".unsorted.bed", "wb") as f:
        f.write(bed_bytes(c[perm], s[perm], e[perm]))


def write_corpus(tmp, n_files, per_file, n_universe, chunk=50):
    """The universe BED file (token id = line) and the query files; returns (universe path, plain query paths)."""
    from gtars_b200 import synth
    u = synth.make_universe(n_universe)
    upath = os.path.join(tmp, "universe.bed")
    with open(upath, "wb") as f:
        f.write(bed_bytes(u["chr"].numpy(), u["start"].numpy(), u["end"].numpy()))
    paths = [os.path.join(tmp, f"q{i:05d}.bed") for i in range(n_files)]
    with Pool(max(1, min(32, os.cpu_count() or 1))) as pool:
        for f0 in range(0, n_files, chunk):
            k = min(chunk, n_files - f0)
            q = synth.make_query_files(u, k, per_file, first_file=f0)
            c, s, e = (q[x].numpy() for x in ("chr", "start", "end"))
            pool.map(write_file, [(paths[f0 + i], c[i * per_file:(i + 1) * per_file], s[i * per_file:(i + 1) * per_file],
                                   e[i * per_file:(i + 1) * per_file], f0 + i) for i in range(k)])
    return upath, paths


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--files", type=int, default=1000)
    ap.add_argument("--regions", type=int, default=100_000, help="regions per file")
    ap.add_argument("--universe", type=int, default=1_000_000, help="peaks of the tokenizer's universe")
    ap.add_argument("--reps", type=int, default=3, help="timed repetitions per arm (best is reported)")
    ap.add_argument("--out", help="also append the JSON lines to this file")
    ap.add_argument("--write-only", action="store_true", help="write the corpus, print its size and stop")
    args = ap.parse_args()
    tmp = tempfile.mkdtemp(prefix="tok_bed_files_")
    out = open(args.out, "a") if args.out else None
    gpu = power = None

    def emit(**kv):
        if gpu is not None:
            kv.update(gpu=gpu, power_limit=power)
        print(json.dumps(kv), flush=True)
        if out:
            out.write(json.dumps(kv) + "\n")
            out.flush()

    try:
        t = time.perf_counter()
        upath, paths = write_corpus(tmp, args.files, args.regions, args.universe)
        forms = {"plain": paths, "gzip": [p + ".gz" for p in paths], "unsorted": [p[:-4] + ".unsorted.bed" for p in paths]}
        emit(workload="write_files", files=args.files, per_file=args.regions, universe=args.universe, wall_s=time.perf_counter() - t,
             file_bytes={k: sum(os.path.getsize(p) for p in v) for k, v in forms.items()})
        if args.write_only:
            return
        gpu, power = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                                    text=True, check=True).stdout.splitlines()[0].split(", ")
        from gtars_b200 import api
        api.device(0)
        tok = api.Tokenizer(upath)
        for form, ps in forms.items():
            cache(ps)
            size = sum(os.path.getsize(p) for p in ps)
            tok.encode_bed_files(ps[:2])                                     # warm-up: modules, allocator, pinned blocks
            arms = (("host_parse_encode_batch", lambda: tok.encode_batch(ps)),
                    ("encode_bed_file_per_file", lambda: [tok.encode_bed_file(p) for p in ps]),
                    ("encode_bed_files", lambda: tok.encode_bed_files(ps)))
            want = None
            for arm, fn in arms:
                dt, got = timed(fn, reps=args.reps)
                if want is None:
                    want = got
                assert got == want, (form, arm)
                emit(workload="tokenize_bed_files", files=args.files, per_file=args.regions, universe=args.universe, format=form,
                     file_bytes=size, arm=arm, wall_s=dt, ids=sum(len(x) for x in got), equal=True)
    finally:
        if out:
            out.close()
        shutil.rmtree(tmp, ignore_errors=True)


if __name__ == "__main__":
    main()
