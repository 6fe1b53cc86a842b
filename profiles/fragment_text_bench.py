"""Wall time of tokenize_fragment_file with the host parse vs device_parse=True, files already in the page cache, plus the
single-window cost of gtgpu_tokenize_fragments_text for two builds of the library timed alternately.

    python profiles/fragment_text_bench.py [--scale 1.0] [--out profiles/fragment_text_bench.jsonl] [--lib PATH ...]

Workloads (at --scale 1), against a 1 M-region universe: one file of 1e8 fragments as plain text and as BGZF (host parse
and device parse); one plain file of 1.1e8 fragments (> 4 GiB), device only; gtgpu_tokenize_fragments_text on 2.5e7
fragments (one window) through each library given with --lib (default: the in-tree one), in alternating child processes,
so that the parent commit's library and this one are timed in the same run.  One JSON line per measurement, each with the
card's name and power limit read in the same run.  Files go to a temporary directory that is removed at the end.
"""
from __future__ import annotations

import argparse
import json
import os
import shutil
import subprocess
import sys
import tempfile
import zlib
from multiprocessing import Pool

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "profiles"))

from score_text_bench import cache, timed, write_fragments  # noqa: E402


def one_window(text_path, reps):
    """Child process: GTGPU_LIB is set by the parent; best wall time of gtgpu_tokenize_fragments_text on the text."""
    import ctypes
    from gtars_b200 import ffi, synth
    exported = ctypes.CDLL(ffi.LIB_PATH)
    for name in [n for n in ffi.SIGNATURES if not hasattr(exported, n)]:  # an older build lacks entry points added since
        del ffi.SIGNATURES[name]
    u = synth.make_universe(1_000_000)
    offs = u["chrom_offsets"].numpy().astype(np.uint64)
    s, e, v = (u[k].numpy().view(np.uint32) for k in ("g_start", "g_end", "g_val"))
    ctx = ffi.Context(0)
    ix = ffi.Index(ctx, ffi.KIND_BITS, offs, s, e, v)
    text = open(text_path, "rb").read()
    names, unk = synth.CHROM_NAMES, int(u["unk_id"])
    ix.tokenize_fragments_text(text, names, unk)                          # warm-up: modules, scratch, pinned cache
    t, (b, o, i) = timed(lambda: ix.tokenize_fragments_text(text, names, unk), reps=reps)
    print(json.dumps(dict(wall_s=t, barcodes=len(b), ids=int(len(i)), ids_sum=int(i.sum(dtype=np.uint64)),
                          names_crc=zlib.crc32("\n".join(b).encode()))))
    ix.close()
    ctx.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--scale", type=float, default=1.0)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "fragment_text_bench.jsonl"))
    ap.add_argument("--lib", action="append", help="libgtars_gpu.so to time at one window (repeatable; default: in-tree)")
    ap.add_argument("--rounds", type=int, default=3, help="alternating rounds of the one-window comparison")
    ap.add_argument("--no-host", action="store_true", help="skip the host-parse arms")
    ap.add_argument("--only-window", action="store_true", help="run the one-window comparison only")
    ap.add_argument("--one-window", help=argparse.SUPPRESS)                # child mode: text path
    args = ap.parse_args()
    if args.one_window:
        one_window(args.one_window, 3)
        return
    from gtars_b200 import api, synth
    gpu, power = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                                text=True, check=True).stdout.splitlines()[0].split(", ")
    tmp = tempfile.mkdtemp(prefix="fragment_text_")
    out = open(args.out, "a")

    def emit(**kv):
        kv.update(gpu=gpu, power_limit=power, scale=args.scale)
        print(json.dumps(kv), flush=True)
        out.write(json.dumps(kv) + "\n")
        out.flush()

    try:
        pool = Pool(max(1, min(32, os.cpu_count() or 1)))
        if not args.only_window:
            u = synth.make_universe(1_000_000)
            uc, us, ue = (u[k].numpy() for k in ("chr", "start", "end"))
            uni = os.path.join(tmp, "universe.bed")
            with open(uni, "w") as f:
                f.write("".join(f"{synth.CHROM_NAMES[c]}\t{s}\t{e}\n" for c, s, e in zip(uc, us, ue)))
            tok = api.Tokenizer(uni)

            # ---- one file of 1e8 fragments, plain and BGZF ----
            n = int(100_000_000 * args.scale)
            path = os.path.join(tmp, "frags.tsv")
            write_fragments(path, n, 31, 1_000_000, pool)
            for fmt, p in (("plain", path), ("bgzf", path + ".gz")):
                cache([p])
                td, dd = timed(lambda: api.tokenize_fragment_file(p, tok, device_parse=True))
                emit(workload="tokenize_fragment_file", fragments=n, format=fmt, file_bytes=os.path.getsize(p), arm="device_parse",
                     wall_s=td, barcodes=len(dd))
                if not args.no_host:
                    th, dh = timed(lambda: api.tokenize_fragment_file(p, tok))
                    emit(workload="tokenize_fragment_file", fragments=n, format=fmt, file_bytes=os.path.getsize(p), arm="host_parse",
                         wall_s=th, equal=dd == dh)
                    del dh
                del dd
            os.remove(path)
            os.remove(path + ".gz")

            # ---- > 4 GiB of plain text, device only ----
            n_big = int(110_000_000 * args.scale)
            big = os.path.join(tmp, "big.tsv")
            write_fragments(big, n_big, 8, 1_000_000)
            cache([big])
            td, dd = timed(lambda: api.tokenize_fragment_file(big, tok, device_parse=True))
            emit(workload="tokenize_fragment_file_big", fragments=n_big, format="plain", file_bytes=os.path.getsize(big),
                 arm="device_parse", wall_s=td, barcodes=len(dd))
            del dd
            os.remove(big)

        # ---- gtgpu_tokenize_fragments_text at one window, libraries alternating ----
        n_one = int(25_000_000 * args.scale)
        one = os.path.join(tmp, "one.tsv")
        write_fragments(one, n_one, 12, 100_000)
        libs = args.lib or [os.path.join(ROOT, "gtars_b200", "libgtars_gpu.so")]
        for r in range(args.rounds):
            for lib in libs:
                env = dict(os.environ, GTGPU_LIB=os.path.abspath(lib))
                res = subprocess.run([sys.executable, os.path.abspath(__file__), "--one-window", one], env=env, capture_output=True,
                                     text=True, check=True)
                emit(workload="tokenize_fragments_text_one_window", fragments=n_one, text_bytes=os.path.getsize(one), lib=lib, round=r,
                     **json.loads(res.stdout.strip().splitlines()[-1]))
        pool.close()
    finally:
        out.close()
        shutil.rmtree(tmp, ignore_errors=True)


if __name__ == "__main__":
    main()
