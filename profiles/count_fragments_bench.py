"""Wall time of count_fragments_by_barcode with the host parse (device_parse=False: the file parsed on one host core, tokenized on
the device, counted into a std::map per barcode) vs device_parse=True (gtgpu_count_fragments_file / _gz: parsed, tokenized and
counted on the device), files already in the page cache.

    python profiles/count_fragments_bench.py [--fragments 100000000] [--formats plain,bgzf] [--reps 3] [--out PATH]

Workload: one seeded file of --fragments fragments (gtars_b200.synth, 40-byte lines, 10^6 barcodes) as plain text and as BGZF,
against a tokenizer over a 10^6-region synth universe file.  Each arm is the whole host-library call from the path to the
per-barcode (token, count) lists (gth_tokenizer_count_fragments[_device]), best of --reps; the conversion of those lists into
Python dicts, the same for both arms, is left out.  The two answers are asserted equal (barcode names and order, every
barcode's token ids and counts).  One JSON line per measurement, each with the card's name and power limit read in the same run.
Files go to a temporary directory that is removed at the end.
"""
from __future__ import annotations

import argparse
import ctypes as C
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

from score_text_bench import cache, write_fragments  # noqa: E402


def lists_arrays(L, h):
    """A gth lists handle as (names, lengths, concatenated interleaved (token, count) pairs); frees the handle."""
    try:
        n = L.gth_lists_n(h)
        names = [L.gth_lists_name(h, i) for i in range(n)]
        lens = np.fromiter((L.gth_lists_len(h, i) for i in range(n)), dtype=np.int64, count=n)
        flat = np.empty(int(lens.sum()), dtype=np.uint32)
        pos = 0
        for i, k in enumerate(lens):
            if k:
                C.memmove(flat.ctypes.data + 4 * pos, L.gth_lists_data(h, i), 4 * int(k))
            pos += int(k)
        return names, lens, flat
    finally:
        L.gth_lists_free(h)


def best_call(L, fn, tok, path, reps):
    """best wall time of fn(tokenizer, path) over reps calls, and the last call's result as arrays"""
    best, h = None, None
    for _ in range(reps):
        if h:
            L.gth_lists_free(h)
        t = time.perf_counter()
        h = fn(tok._h, os.fsencode(path))
        dt = time.perf_counter() - t
        if not h:
            raise RuntimeError(L.gth_last_error().decode())
        best = dt if best is None else min(best, dt)
    return best, lists_arrays(L, h)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--fragments", type=int, default=100_000_000)
    ap.add_argument("--universe", type=int, default=1_000_000)
    ap.add_argument("--barcodes", type=int, default=1_000_000)
    ap.add_argument("--formats", default="plain,bgzf")
    ap.add_argument("--reps", type=int, default=3, help="timed calls per arm (best is reported)")
    ap.add_argument("--out", help="also append the JSON lines to this file")
    args = ap.parse_args()
    from gtars_b200 import api, synth
    gpu, power = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                                text=True, check=True).stdout.splitlines()[0].split(", ")
    tmp = tempfile.mkdtemp(prefix="count_fragments_")
    out = open(args.out, "a") if args.out else None

    def emit(**kv):
        kv.update(gpu=gpu, power_limit=power)
        print(json.dumps(kv), flush=True)
        if out:
            out.write(json.dumps(kv) + "\n")
            out.flush()

    try:
        formats = args.formats.split(",")
        t = time.perf_counter()
        u = synth.make_universe(args.universe)
        uc, us, ue = (u[k].numpy() for k in ("chr", "start", "end"))
        uni = os.path.join(tmp, "universe.bed")
        with open(uni, "w") as f:
            f.write("".join(f"{synth.CHROM_NAMES[c]}\t{s}\t{e}\n" for c, s, e in zip(uc, us, ue)))
        path = os.path.join(tmp, "frags.tsv")
        with Pool(max(1, min(32, os.cpu_count() or 1))) as pool:
            write_fragments(path, args.fragments, 47, args.barcodes, pool if "bgzf" in formats else None)
        emit(workload="write_files", fragments=args.fragments, wall_s=time.perf_counter() - t)
        L = api.lib()
        api.device(0)
        tok = api.Tokenizer(uni)
        for fmt in formats:
            p = path if fmt == "plain" else path + ".gz"
            cache([p])
            best_call(L, L.gth_tokenizer_count_fragments_device, tok, p, 1)  # warm-up: modules, scratch, pinned blocks
            td, dev = best_call(L, L.gth_tokenizer_count_fragments_device, tok, p, args.reps)
            th, host = best_call(L, L.gth_tokenizer_count_fragments, tok, p, args.reps)
            equal = dev[0] == host[0] and np.array_equal(dev[1], host[1]) and np.array_equal(dev[2], host[2])
            assert equal, fmt
            base = dict(workload="count_fragments_by_barcode", fragments=args.fragments, universe=args.universe, format=fmt,
                        file_bytes=os.path.getsize(p), barcodes=len(dev[0]), entries=int(len(dev[2]) // 2), reps=args.reps, equal=equal)
            emit(**base, arm="host_parse", wall_s=th)
            emit(**base, arm="device_parse", wall_s=td, speedup=th / td)
            del dev, host
    finally:
        if out:
            out.close()
        shutil.rmtree(tmp, ignore_errors=True)


if __name__ == "__main__":
    main()
