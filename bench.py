#!/usr/bin/env python
"""bench.py — headline benchmark: tokenize synthetic hg38-shaped BED files against a 1 M-region universe.

A "step" is one pass of the hot path (Tokenizer::encode for every file, gtars-tokenizers/src/tokenizer.rs:140-171)
over BASELINE.json configs[1] (C2): 10 000 files x 100 000 regions = 1e9 query intervals vs a 1 M-region universe.

  value     query intervals / s, device-resident inputs, CUDA events around K back-to-back steps (max over ranks)
  e2e       the same metric through the C-ABI host entry point gtgpu_tokenize_files_packed (--e2e-api: packed / compact /
            runs) with PINNED HOST buffers, H2D of the queries and D2H of the ids inside the timed region; `marshal` = the
            host-side packing of the caller's flat (chr, start, end) arrays into that wire format, timed separately;
            `pcie` = what concurrent pinned H2D + D2H copies reach on this box (the ceiling of any e2e number)
  roofline  algorithmic HBM bytes of the fused kernel / its own CUDA-event time, vs MEASURED_PEAKS.json hbm_gbs
  cpu_baseline  the CPU oracle (C++ restatement of the reference's algorithm; the reference is Rust and cannot be
            built here) on a bounded sample of the same files, 1 thread (the reference path is single-threaded)
  parity    every id and per-file offset of >= 10 % of the files compared with the multithreaded oracle (untimed)
  configs   sub-records for BASELINE.json configs[2..4], each sharded over the N ranks as the config says, with its own
            timing, algorithmic bytes, roofline fraction and a parity check of the full-size result against the oracle:
              c3  Bits count, 100 M queries vs a 50 M-interval database, query-sharded (strong scaling)
              c4  LOLA region-hit matrix, 1 k user sets x 10 k database sets, database sharded by set + ncclAllGather
              c5  fragment tokenization, 1 B unsorted fragments vs the 1 M-peak universe, fragment-sharded
              backend  the headline workload (a tenth of the files) on the other overlapper backend (AIList when C2 runs Bits)
              gz  a bgzip'ed BED file inflated on the device (one warp per member) and tokenized, vs zlib on one host thread

`--scaling weak` (default): every rank owns `--files` files (1e9 queries per GPU); `--scaling strong`: `--files` files in
total.  `--impl reference` times the oracle with all host threads instead (rank 0 only).  Multi-GPU (torchrun): files
are sharded across ranks (rank r owns files [r*F, (r+1)*F)), universe replicated, no collective on the C2 data path.

`--dump-outputs DIR` writes rank 0's C2 result of the last timed step as float64 .npy files: token_ids.npy and
file_token_offsets.npy (raw per-file offsets into the ids, before the per-file [unk] rule).  An array longer than
DUMP_MAX_VALUES is written as a fixed, seeded sample, with the sampled positions in <name>_positions.npy.  The inputs are
counter-based (gtars_b200/synth.py), so the same arguments give the same files on every run and every build.
"""
from __future__ import annotations

import argparse
import ctypes as C
import hashlib
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time
import traceback

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "query_intervals_per_sec_tokenize_vs_universe"
UNIT = "queries/s"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--files", type=int, default=10_000, help="files per GPU (weak scaling) or in total (strong scaling)")
    ap.add_argument("--per-file", type=int, default=100_000)
    ap.add_argument("--universe", type=int, default=1_000_000)
    ap.add_argument("--kind", default="bits", choices=["bits", "ailist"])
    ap.add_argument("--nested", type=float, default=0.0, help="fraction of wide intervals (C2n variant)")
    ap.add_argument("--width-scale", type=int, default=1, help="multiply the 200-600 bp query widths (wide-query variant)")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"])
    ap.add_argument("--cpu-seconds", type=float, default=10.0, help="budget of the cpu_baseline leg")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--e2e-api", default="packed", choices=["packed", "compact", "runs"], help="host entry point of the e2e leg")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--configs", default="backend,gz,c3,c4,c5", help="sub-records to add (comma separated; empty = none)")
    ap.add_argument("--sub-scale", type=float, default=1.0, help="scale factor on the sizes of the c3/c4/c5 sub-records")
    ap.add_argument("--parity-files", type=int, default=1000, help="files of the full-size C2 result checked against the oracle")
    ap.add_argument("--no-pcie-probe", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write rank 0's result of the last timed step (token ids and per-file "
                                                          "token offsets) to DIR/<name>.npy as float64, for output-by-output "
                                                          "comparison of two builds")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


def workload_config(args, world):
    per_gpu = args.files if args.scaling == "weak" else args.files // world
    return {
        "workload": f"C2: tokenize {per_gpu} files x {args.per_file} regions per GPU vs {args.universe}-region hg38 universe",
        "files_per_gpu": per_gpu, "regions_per_file": args.per_file, "universe_regions": args.universe,
        "backend": args.kind, "nested_frac": args.nested, "query_width_scale": args.width_scale,
        "sharding": f"files x{world} (universe replicated)", "scaling": args.scaling,
        "l2_policy": "inputs (12 B/query x 1e9) are far larger than the 126 MB L2; no flush needed",
    }


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def host_threads() -> int:
    """CPUs this process may run on — NOT OMP_NUM_THREADS, which torch.distributed.run pins to 1 for its workers."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return max(1, os.cpu_count() or 1)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 100 ms while the timed region runs."""
    FIELDS = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
              "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits",
                                       "-i", str(self.gpu), "-lms", "100"], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.f.read().splitlines():
            parts = [x.strip() for x in line.split(",")]
            if len(parts) < 9:
                continue
            try:
                sm.append(float(parts[1]))
                mx.append(float(parts[2]))
            except ValueError:
                continue
            for name, val in zip(names, parts[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        os.unlink(self.f.name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def oracle_index(args, universe):
    from oracle import oracle as orc
    offs = universe["chrom_offsets"].cpu().numpy().astype(np.uint64)
    s, e, v = (universe[k].cpu().numpy().view(np.uint32) for k in ("g_start", "g_end", "g_val"))
    return orc.Index(orc.BITS if args.kind == "bits" else orc.AILIST, offs, s, e, v)


def cpu_oracle_rate(args, threads, seconds, universe):
    """Oracle tokenize throughput on files [0, k) of the same synthetic stream; k grows until `seconds` are spent."""
    from gtars_b200 import synth
    ix = oracle_index(args, universe)
    batch = max(1, min(args.files, (4 if threads == 1 else 4 * threads)))
    done_q, spent, first = 0, 0.0, 0
    while spent < seconds and first < args.files:
        nf = min(batch, args.files - first)
        q = synth.make_query_files(universe, nf, args.per_file, first_file=first, width_scale=args.width_scale)
        qc, qs, qe = (q[k].numpy().view(np.uint32) for k in ("chr", "start", "end"))
        fo = q["file_offsets"].numpy().astype(np.uint64)
        t0 = time.perf_counter()
        ix.tokenize_files(fo, qc, qs, qe, universe["unk_id"], threads=threads)
        spent += time.perf_counter() - t0
        done_q += len(qc)
        first += nf
    return done_q / spent, f"files [0,{first}) = {done_q} queries in {spent:.2f} s"


def run_reference(args, rank, world):
    """The reference arm: the CPU oracle (a C++ port; the Rust reference cannot be compiled in this image) with every
    host thread, on the same bounded sample of the workload per step at every N (rank 0 alone runs it)."""
    if rank != 0:
        return
    from gtars_b200 import synth
    threads = host_threads()
    u = synth.make_universe(args.universe, nested_frac=args.nested)
    ix = oracle_index(args, u)
    sample_files = min(args.files, 128)
    q = synth.make_query_files(u, sample_files, args.per_file, width_scale=args.width_scale)
    qc, qs, qe = (q[k].numpy().view(np.uint32) for k in ("chr", "start", "end"))
    fo = q["file_offsets"].numpy().astype(np.uint64)
    for _ in range(max(args.warmup, 1)):
        ix.tokenize_files(fo, qc, qs, qe, u["unk_id"], threads=threads)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        ix.tokenize_files(fo, qc, qs, qe, u["unk_id"], threads=threads)
    dt = (time.perf_counter() - t0) / args.steps
    value = len(qc) / dt
    sample = f"{sample_files} files x {args.per_file} regions per step (bounded sample of the workload; the same at every N)"
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": args.scaling,
        "vs_baseline": None, "dtype": "u32", "data": "synthetic", "config": workload_config(args, world),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample,
                         "note": "C++ restatement of gtars' algorithm on all host threads (OpenMP over files); the Rust "
                                 "reference is single-threaded on this path and cannot be built in this image"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }))


# --dump-outputs: an array longer than this is dumped as a fixed, seeded sample of its positions, and the sorted positions
# are dumped beside it; ids + positions + offsets + positions stay under 64 MB of float64 (exact for u32 ids and offsets < 2^53).
DUMP_MAX_VALUES = 1 << 20


def dump_positions(n: int, seed: int):
    """None when all n values fit the dump, else DUMP_MAX_VALUES distinct sorted positions of [0, n), the same on every run."""
    if n <= DUMP_MAX_VALUES:
        return None
    return np.sort(np.random.default_rng(seed).choice(n, DUMP_MAX_VALUES, replace=False))


def write_dump(out_dir: str, arrays: dict):
    """arrays: name -> (values, positions or None); everything is written as float64."""
    os.makedirs(out_dir, exist_ok=True)
    for name, (values, pos) in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), np.asarray(values).astype(np.float64))
        if pos is not None:
            np.save(os.path.join(out_dir, f"{name}_positions.npy"), pos.astype(np.float64))


def digest64(*arrays) -> str:
    h = hashlib.blake2b(digest_size=8)
    for a in arrays:
        h.update(np.ascontiguousarray(a).tobytes())
    return h.hexdigest()


class Dist:
    """torch.distributed plumbing: NCCL for the device-side reductions of timings, gloo for host-side waits."""

    def __init__(self, torch, world, dev):
        self.torch, self.world, self.dev = torch, world, dev
        self.dist = None
        if world > 1:
            import torch.distributed as dist
            self.dist = dist
            dist.init_process_group("nccl", device_id=dev)
            self.cpu_group = dist.new_group(backend="gloo")  # host-side waits that keep the waiting ranks off their GPUs

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()

    def host_barrier(self):
        """Barrier on the CPU (gloo): ranks waiting here launch nothing on their GPU (an NCCL barrier spins a kernel)."""
        if self.world > 1:
            self.dist.barrier(group=self.cpu_group)

    def _reduce(self, x, op):
        if self.world == 1:
            return x
        t = self.torch.tensor([x], dtype=self.torch.float64, device=self.dev)
        self.dist.all_reduce(t, op=op)
        return float(t.item())

    def max(self, x):
        return self._reduce(x, self.dist.ReduceOp.MAX) if self.world > 1 else x

    def sum(self, x):
        return self._reduce(x, self.dist.ReduceOp.SUM) if self.world > 1 else x

    def gather_objects(self, obj):
        if self.world == 1:
            return [obj]
        out = [None] * self.world
        self.dist.all_gather_object(out, obj)
        return out

    def close(self):
        if self.world > 1:
            self.dist.destroy_process_group()


def pcie_probe(torch, dev, D, h2d_bytes, d2h_bytes):
    """Concurrent pinned H2D + D2H copies on every rank at once, in the byte mix of one e2e step (a quarter of its bytes, in
    pipeline-sized pieces): what the box's PCIe / host fabric delivers to this traffic pattern — the floor of any e2e time."""
    piece = 192 << 20
    n_in = max(1, int(h2d_bytes / 4 / piece))
    out_piece = max(1 << 20, int(piece * d2h_bytes / max(h2d_bytes, 1)))
    h_in = torch.empty(piece, dtype=torch.uint8, pin_memory=True)
    h_out = torch.empty(out_piece, dtype=torch.uint8, pin_memory=True)
    d_in = torch.empty(piece, dtype=torch.uint8, device=dev)
    d_out = torch.zeros(out_piece, dtype=torch.uint8, device=dev)
    s_in, s_out = torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)

    def run(do_in, do_out):
        torch.cuda.synchronize()
        D.barrier()
        t0 = time.perf_counter()
        for _ in range(n_in):
            if do_in:
                with torch.cuda.stream(s_in):
                    d_in.copy_(h_in, non_blocking=True)
            if do_out:
                with torch.cuda.stream(s_out):
                    h_out.copy_(d_out, non_blocking=True)
        s_in.synchronize()
        s_out.synchronize()
        return D.max(time.perf_counter() - t0)

    run(True, True)
    t_in, t_out = run(True, False), run(False, True)
    t_mix = min(run(True, True), run(True, True))
    b_in, b_out = n_in * piece, n_in * out_piece
    out = {"h2d_alone_gbs_per_gpu": b_in / t_in / 1e9, "d2h_alone_gbs_per_gpu": b_out / t_out / 1e9,
           "mixed_h2d_gbs_per_gpu": b_in / t_mix / 1e9, "mixed_d2h_gbs_per_gpu": b_out / t_mix / 1e9,
           "aggregate_mixed_gbs": (b_in + b_out) * D.world / t_mix / 1e9, "gpus_copying_at_once": D.world,
           "floor_ms_for_one_e2e_step": t_mix * (h2d_bytes / b_in) * 1e3,
           "note": f"{n_in} x ({piece >> 20} MiB in + {out_piece >> 20} MiB out) pinned copies on two streams, all ranks at the "
                   "same time, slowest rank; the mix is the e2e step's own H2D : D2H ratio"}
    del h_in, h_out, d_in, d_out
    return out


# =====================================================================================================================
# sub-records: BASELINE.json configs[2..4]
# =====================================================================================================================
def sub_c3(args, torch, dev, ctx, stream, D, rank, world, peak):
    """C3: Bits::count (bits.rs:337-344) of 100 M unsorted queries against a 50 M-interval database; the queries are
    sharded over the ranks in contiguous blocks, the database is replicated (strong scaling)."""
    from gtars_b200 import ffi, shard, synth
    from oracle import oracle as orc
    n_db, n_q_total = int(50_000_000 * args.sub_scale), int(100_000_000 * args.sub_scale)
    q0, q1 = shard.block_range(n_q_total, world, rank)
    n_q = q1 - q0
    t0 = time.perf_counter()
    db = synth.make_uniform_intervals(n_db, synth.SEED_LOLA_DB, device=dev, min_w=100, max_w=10_000)
    g = synth.group_by_chrom(db["chr"], db["start"], db["end"])
    offs = g["chrom_offsets"].cpu().numpy().astype(np.uint64)
    s, e = (g[k].cpu().numpy().view(np.uint32) for k in ("g_start", "g_end"))
    del db, g
    t1 = time.perf_counter()
    ix = ffi.Index(ctx, ffi.KIND_BITS, offs, s, e)
    build_s = time.perf_counter() - t1
    q = synth.make_uniform_intervals(n_q, synth.SEED_QUERIES, device=dev, min_w=100, max_w=2000, log_uniform=False, first=q0)
    d_out = torch.empty(n_q, dtype=torch.int32, device=dev)
    fn = lambda: ix.count_dev(n_q, q["chr"].data_ptr(), q["start"].data_ptr(), q["end"].data_ptr(), 0, d_out.data_ptr())
    with torch.cuda.stream(stream):
        for _ in range(3):
            fn()
        stream.synchronize()
        D.barrier()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = ctx.launch_count()
        ev0.record(stream)
        for _ in range(args.steps):
            fn()
        ev1.record(stream)
        stream.synchronize()
        launches = (ctx.launch_count() - l0) // args.steps
    ms = D.max(ev0.elapsed_time(ev1) / args.steps)
    # parity: the queries of this rank's first 4 M that fall on chr1 / chr21 / chrX, against the C++ oracle built over
    # exactly those chromosomes of the database (Bits::count depends on the query's chromosome only)
    parity = None
    m = min(n_q, 4_000_000)
    chroms = [0, 20, 22]
    qc, qs, qe = (q[k][:m].cpu().numpy().view(np.uint32) for k in ("chr", "start", "end"))
    sel = np.isin(qc, chroms)
    keep = np.zeros(len(offs) - 1, dtype=bool)
    keep[chroms] = True
    sub_counts = np.where(keep, np.diff(offs.astype(np.int64)), 0)
    sub_offs = np.concatenate([[0], np.cumsum(sub_counts)]).astype(np.uint64)
    idx = np.concatenate([np.arange(int(offs[c]), int(offs[c + 1])) for c in chroms])
    o = orc.Index(orc.BITS, sub_offs, s[idx], e[idx])
    want = o.count(qc[sel], qs[sel], qe[sel], threads=host_threads())
    got = d_out[:m].cpu().numpy().view(np.uint32)[sel]
    parity = bool(np.array_equal(got, want))
    parity_all = all(D.gather_objects(parity))
    checked = int(D.sum(float(sel.sum())))
    algo = 16 * n_q_total + 8 * n_db  # SURVEY 8d: 12 B query + 4 B count per query, 8 B per database interval (read once)
    info = ix.info()
    ix.close()
    del q, d_out
    return {"workload": f"C3: Bits count, {n_q_total} unsorted queries vs a {n_db}-interval database", "scaling": "strong",
            "sharding": f"queries in {world} contiguous blocks, database replicated, no collective",
            "queries_total": n_q_total, "queries_per_gpu": n_q, "db_intervals": n_db, "ms": ms,
            "value": n_q_total / (ms * 1e-3), "unit": "queries/s", "algorithmic_bytes": algo,
            "frac": (16 * n_q + 8 * n_db) / (ms * 1e-3) / 1e9 / peak,
            "frac_note": "per GPU: (16 B x its queries + 8 B x database) / time / measured HBM peak",
            "kernels_per_step": launches, "index_build_s": build_s, "data_gen_s": t1 - t0,
            "parity_vs_oracle": parity_all, "parity_queries_checked": checked, "index": info}


def sub_c4(args, torch, dev, ctx, stream, D, rank, world, peak):
    """C4: run_lola's count step (enrichment.rs:198-211): region-hit matrix of 1 k user sets + the universe against a
    10 k-set database, the database sharded by region set over the ranks, one ncclAllGather of the column blocks."""
    from gtars_b200 import ffi, shard, synth
    from oracle import oracle as orc
    n_db = max(int(10_000 * args.sub_scale), 8 * world)
    per_db, n_user, per_user = 20_000, max(int(1000 * args.sub_scale), 4), 10_000
    lo, hi = shard.db_set_range(n_db, world, rank)
    t0 = time.perf_counter()
    db = synth.make_uniform_intervals((hi - lo) * per_db, synth.SEED_LOLA_DB, device=dev, min_w=200, max_w=5000, first=lo * per_db)
    dfo = (np.arange(hi - lo + 1) * per_db).astype(np.uint64)
    dc, ds, de = (db[k].cpu().numpy().view(np.uint32) for k in ("chr", "start", "end"))
    del db
    t1 = time.perf_counter()
    g = ffi.Igd(ctx, dfo, synth.N_CHROMS, dc, ds, de)
    build_s = time.perf_counter() - t1
    if world > 1:
        shard.init_comm_from_torch(ctx)
    u = synth.make_universe(1_000_000, device=dev)
    pick = synth.rand_u63(synth.SEED_LOLA_USER, 1, torch.arange(n_user * per_user, device=dev)) % u["n"]
    n_univ = int(u["n"])
    n_q = n_user * per_user + n_univ
    # the caller's arrays and the result matrix live in pinned host memory, so the copies inside the call are DMA
    qc, qs, qe = (ffi.pinned_empty(n_q, np.uint32) for _ in range(3))
    for dst, a, b in ((qc, u["chr"][pick], u["chr"]), (qs, u["start"][pick], u["start"]), (qe, u["end"][pick], u["end"])):
        torch.from_numpy(dst.view(np.int32)).copy_(torch.cat([a, b]))
    torch.cuda.synchronize()
    so = np.concatenate([np.arange(n_user + 1) * per_user, [n_user * per_user + n_univ]]).astype(np.uint64)
    h_out = ffi.pinned_empty((n_user + 1) * n_db, np.uint64).reshape(n_user + 1, n_db)
    call = lambda: g.count_sharded(True, n_db, so, qc, qs, qe, 1, out=h_out)
    call()
    call()
    ctx.timing_enable(True)
    D.barrier()
    l0 = ctx.launch_count()
    t2 = time.perf_counter()
    for _ in range(args.steps):
        hits = call()
    ms = D.max((time.perf_counter() - t2) / args.steps * 1e3)
    launches = (ctx.launch_count() - l0) // args.steps
    k_ms = ctx.timing_read()
    ctx.timing_enable(False)
    kernel_ms = D.max(statistics.mean(k_ms) if k_ms else 0.0)
    # parity on full-size output: columns are independent (a set's counts depend on that set's records only), so the
    # oracle builds an IGD over 2 database sets of every rank's shard and must reproduce those columns for the first
    # 3 user sets and a slice of the universe — which also checks where the all-gather put every rank's block
    k = 3
    u_lo = n_user * per_user
    sel = np.concatenate([np.arange(k * per_user), np.arange(u_lo, u_lo + 200_000)])
    sso = np.concatenate([np.arange(k + 1) * per_user, [k * per_user + 200_000]]).astype(np.uint64)
    got_slice = g.count_sharded(True, n_db, sso, qc[sel], qs[sel], qe[sel], 1)  # collective: every rank calls it
    parity = None
    if rank == 0:
        cols = sorted({c for r in range(world) for c in (shard.db_set_range(n_db, world, r)[0], shard.db_set_range(n_db, world, r)[1] - 1)})
        parts = [synth.make_uniform_intervals(per_db, synth.SEED_LOLA_DB, min_w=200, max_w=5000, first=c * per_db) for c in cols]
        oc = np.concatenate([p["chr"].numpy().view(np.uint32) for p in parts])
        os_ = np.concatenate([p["start"].numpy().view(np.uint32) for p in parts])
        oe = np.concatenate([p["end"].numpy().view(np.uint32) for p in parts])
        o = orc.Igd((np.arange(len(cols) + 1) * per_db).astype(np.uint64), oc, os_, oe)
        want = o.count_region_hits(sso, qc[sel], qs[sel], qe[sel], 1, threads=host_threads())
        parity = bool(np.array_equal(hits[:k][:, cols], want[:k]) and np.array_equal(got_slice[:, cols], want))
        tables = orc.lola_tables(hits[:n_user], hits[n_user], np.full(n_user, per_user), n_univ)
        parity = parity and tables.shape == (n_user, n_db, 4)
    pair_hits = int(hits.sum())
    algo = 12 * n_q + 12 * n_db * per_db + 8 * (n_user + 1) * n_db
    info = g.info()
    g.close()
    for a in (qc, qs, qe):
        ffi.pinned_free(a)
    return {"workload": f"C4: LOLA region-hit matrix, {n_user} user sets x {per_user} regions + {n_univ}-region universe vs {n_db} database sets x {per_db}",
            "scaling": "strong", "sharding": f"database sharded by region set over {world} ranks, query sets replicated, "
                                             + ("one ncclAllGather of the column blocks" if world > 1 else "single rank: no collective"),
            "db_sets": n_db, "db_sets_per_gpu": hi - lo, "db_records": n_db * per_db, "query_regions": n_q,
            "ms": ms, "ms_note": "whole gtgpu_igd_count_sharded call from / to pinned host memory: H2D of the query sets, count kernel, all-gather, transposition, D2H of the matrix",
            "kernel_ms": kernel_ms, "value": n_q / (ms * 1e-3), "unit": "query regions/s",
            "region_file_hits": pair_hits, "hits_per_s": pair_hits / (ms * 1e-3), "algorithmic_bytes": algo,
            "frac": (12 * n_q + 12 * (hi - lo) * per_db + 8 * (n_user + 1) * n_db) / max(kernel_ms, 1e-9) / 1e6 / peak,
            "frac_note": "count kernel only; atomic / L2-bound by construction, the HBM fraction is low on purpose (SURVEY 8d)",
            "kernels_per_step": launches, "index_build_s": build_s, "data_gen_s": t1 - t0,
            "parity_vs_oracle": parity, "parity_what": "2 database sets of every rank's shard x (3 user sets + 200 k universe regions), all cells",
            "igd_rank0": info}


def sub_c5(args, torch, dev, ctx, stream, D, rank, world, peak, universe, index):
    """C5: tokenize_fragment_file (fragments.rs:12-82) for 1 B unsorted fragments vs the 1 M-peak universe: fragments are
    sharded over the ranks in contiguous blocks; every rank groups its block by barcode on the device (hand-written radix
    sort) — per-barcode lists of the shards concatenate in shard order."""
    from gtars_b200 import ffi, shard, synth
    n_total = int(1_000_000_000 * args.sub_scale)
    n_bc = 100_000
    f0, f1 = shard.block_range(n_total, world, rank)
    n = f1 - f0
    t0 = time.perf_counter()
    d_chr = torch.empty(n, dtype=torch.int32, device=dev)
    d_start = torch.empty(n, dtype=torch.int32, device=dev)
    d_end = torch.empty(n, dtype=torch.int32, device=dev)
    d_bc = torch.empty(n, dtype=torch.int32, device=dev)
    chunk = 1 << 24
    for a in range(0, n, chunk):
        k = min(chunk, n - a)
        # "file" index = position / chunk is only the counter base of the generator: fragments [f0 + a, f0 + a + k)
        q = _fragments(synth, universe, f0 + a, k, dev)
        d_chr[a:a + k], d_start[a:a + k], d_end[a:a + k], d_bc[a:a + k] = q
        del q
    cap = n + n // 4 + 1024
    d_ids = torch.empty(cap, dtype=torch.int32, device=dev)
    d_bco = torch.empty(n_bc + 1, dtype=torch.int64, device=dev)
    d_total = torch.zeros(1, dtype=torch.int64, device=dev)
    torch.cuda.synchronize()
    gen_s = time.perf_counter() - t0
    unk = int(universe["unk_id"])
    fn = lambda: index.tokenize_fragments_dev(n, d_chr.data_ptr(), d_start.data_ptr(), d_end.data_ptr(), d_bc.data_ptr(), n_bc,
                                              unk, d_bco.data_ptr(), d_ids.data_ptr(), cap, d_total.data_ptr())
    with torch.cuda.stream(stream):
        for _ in range(2):
            fn()
        stream.synchronize()
        total = int(d_total.item())
        assert 0 < total <= cap, "C5: id capacity"
        D.barrier()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = ctx.launch_count()
        ev0.record(stream)
        for _ in range(args.steps):
            fn()
        ev1.record(stream)
        stream.synchronize()
        launches = (ctx.launch_count() - l0) // args.steps
    ms = D.max(ev0.elapsed_time(ev1) / args.steps)
    tokens_total = int(D.sum(float(total)))
    # parity on the full-size result: ~200 barcodes' complete lists.  Their fragments are pulled out of this rank's block
    # in input order, the oracle tokenizes them one by one, and each barcode's list must equal the device's list.
    from oracle import oracle as orc
    pick = torch.unique(synth.rand_u63(synth.SEED_FRAGMENTS, 11, torch.arange(200, device=dev)) % n_bc)

    def select(barcodes):
        lut = torch.zeros(n_bc, dtype=torch.bool, device=dev)
        lut[barcodes] = True
        parts = []
        for a in range(0, n, 1 << 26):
            b = min(n, a + (1 << 26))
            parts.append(torch.nonzero(lut[d_bc[a:b].long()]).flatten() + a)
        return torch.cat(parts)

    sel = select(pick)
    if sel.numel() > 3_000_000:
        pick = pick[: max(1, pick.numel() * 3_000_000 // sel.numel())]
        sel = select(pick)
    dense = torch.searchsorted(pick, d_bc[sel].long())
    sc, ss, se = (t[sel].cpu().numpy().view(np.uint32) for t in (d_chr, d_start, d_end))
    o_off, o_ids = oracle_index(args, universe).tokenize_fragments(sc, ss, se, dense.cpu().numpy().astype(np.uint32), int(pick.numel()), unk)
    bco = d_bco.cpu().numpy()
    ok = True
    got_parts = []
    for j, b in enumerate(pick.cpu().numpy()):
        got = d_ids[int(bco[b]):int(bco[b + 1])].cpu().numpy().view(np.uint32)
        got_parts.append(got)
        ok = ok and np.array_equal(got, o_ids[int(o_off[j]):int(o_off[j + 1])])
    ok = ok and int(bco[n_bc]) == total and bool((np.diff(bco) >= 0).all())
    parity_all = all(D.gather_objects(bool(ok)))
    checked = int(D.sum(float(sel.numel())))
    # e2e through the host entry point (pinned host arrays in, pinned result out) on a bounded slice of this rank's block
    m = min(n, 125_000_000)
    h = [ffi.pinned_empty(m, np.uint32) for _ in range(4)]
    for dst, src in zip(h, (d_chr, d_start, d_end, d_bc)):
        torch.from_numpy(dst.view(np.int32)).copy_(src[:m])
    torch.cuda.synchronize()
    L = ffi.lib()
    _, buf = index.tokenize_fragments(h[0], h[1], h[2], h[3], n_bc, unk, keep_buf=True)
    L.gtgpu_buf_free(buf)
    D.barrier()
    t2 = time.perf_counter()
    e_off, buf = index.tokenize_fragments(h[0], h[1], h[2], h[3], n_bc, unk, keep_buf=True)
    e2e_s = D.max(time.perf_counter() - t2)
    e2e_tokens = int(L.gtgpu_buf_len(buf))
    assert e2e_tokens == int(e_off[-1])
    L.gtgpu_buf_free(buf)
    for a in h:
        ffi.pinned_free(a)
    algo = 16 * n + 4 * total + 8 * (n_bc + 1) + 12 * int(universe["n"])
    del d_chr, d_start, d_end, d_bc, d_ids
    return {"workload": f"C5: fragment tokenization, {n_total} unsorted fragments vs the {int(universe['n'])}-peak universe, {n_bc} barcodes",
            "scaling": "strong", "sharding": f"fragments in {world} contiguous blocks, universe replicated, per-barcode lists concatenate in shard order, no collective",
            "fragments_total": n_total, "fragments_per_gpu": n, "tokens_total": tokens_total, "ms": ms,
            "value": n_total / (ms * 1e-3), "unit": "fragments/s", "algorithmic_bytes_per_gpu": algo,
            "frac": algo / (ms * 1e-3) / 1e9 / peak,
            "frac_note": "per GPU: (16 B x fragments + 4 B x tokens + barcode offsets + universe) / time of the whole device-resident "
                         "pipeline (find with barcode tags, two radix passes: pairs -> packed words -> tokens, scans) / measured HBM peak",
            "kernels_per_step": launches, "data_gen_s": gen_s,
            "e2e": {"fragments_per_gpu": m, "seconds": e2e_s, "value": m * world / e2e_s, "unit": "fragments/s",
                    "note": "gtgpu_tokenize_fragments, pinned host arrays in (16 B/fragment), pinned result out; bounded slice of the block",
                    "tokens": e2e_tokens},
            "parity_vs_oracle": parity_all, "parity_fragments_checked": checked, "parity_barcodes": int(pick.numel()),
            "parity_digest": digest64(*got_parts)}


def bgzf_compress(data: bytes, block=60_000, level=6) -> bytes:
    """A BGZF file as bgzip writes it: independent gzip members with the 'BC' extra field (BSIZE) + the empty EOF block."""
    import struct
    import zlib
    out = []
    for a in list(range(0, len(data), block)) + [None]:
        ch = data[a:a + block] if a is not None else b""
        co = zlib.compressobj(level, zlib.DEFLATED, -15)
        body = co.compress(ch) + co.flush()
        out.append(b"\x1f\x8b\x08\x04" + b"\0" * 4 + b"\x00\xff" + struct.pack("<H", 6) + b"BC" + struct.pack("<HH", 2, 12 + 6 + len(body) + 8 - 1)
                   + body + struct.pack("<II", zlib.crc32(ch), len(ch)))
    return b"".join(out)


def sub_gz(args, torch, dev, ctx, stream, D, rank, world, peak, universe, index):
    """SURVEY 8f f4: a bgzip'ed BED file (the reference reads `.gz` through flate2's MultiGzDecoder, gtars-core/src/utils.rs:115-126)
    inflated on the device, one warp per BGZF member, and tokenized without the text ever crossing PCIe.  Rank-local, same file
    on every rank; compared with zlib on one host thread (what the reference's reader does)."""
    import zlib
    import pandas as pd
    from gtars_b200 import ffi, synth
    n_lines = 2_000_000
    q = synth.make_query_files(universe, 20, n_lines // 20, first_file=0)
    names = np.array(list(synth.CHROM_NAMES))
    qc, qs, qe = (q[k].numpy() for k in ("chr", "start", "end"))
    t0 = time.perf_counter()
    text = pd.DataFrame({"c": names[qc], "s": qs, "e": qe}).to_csv(sep="\t", header=False, index=False).encode()
    gz = bgzf_compress(text)
    prep_s = time.perf_counter() - t0
    members = ffi.gzip_members(gz)
    t0 = time.perf_counter()
    z_text = b"".join(zlib.decompress(gz[int(a):int(b)], 31) for a, b in zip(members[:-1], members[1:]))
    zlib_s = time.perf_counter() - t0
    got, _ = ffi.gunzip(ctx, gz, members)   # warm-up + parity
    same_text = got == text and z_text == text
    del got, z_text
    ctx.timing_enable(True)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        ffi.gunzip(ctx, gz, members)
    wall_s = (time.perf_counter() - t0) / args.steps
    k_ms = ctx.timing_read()
    ctx.timing_enable(False)
    kernel_ms = statistics.median(k_ms) if k_ms else None
    unk = int(universe["unk_id"])
    want = index.tokenize_bed(text, list(names), unk)
    ids = index.tokenize_bed_gz(gz, list(names), unk, member_offsets=members)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        index.tokenize_bed_gz(gz, list(names), unk, member_offsets=members)
    tok_s = (time.perf_counter() - t0) / args.steps
    t0 = time.perf_counter()
    for _ in range(args.steps):
        index.tokenize_bed(text, list(names), unk)
    tok_text_s = (time.perf_counter() - t0) / args.steps
    ok = bool(same_text and np.array_equal(ids, want))
    return {"workload": f"bgzip'ed BED file, {n_lines} lines: inflate on the device (one warp per BGZF member) + parse + sort + tokenize",
            "gz_bytes": len(gz), "text_bytes": len(text), "members": int(len(members) - 1),
            "gunzip_kernel_ms": kernel_ms, "gunzip_kernel_text_gbs": (len(text) / (kernel_ms * 1e-3) / 1e9) if kernel_ms else None,
            "gunzip_host_to_host_ms": wall_s * 1e3, "zlib_one_thread_ms": zlib_s * 1e3,
            "tokenize_bed_gz_ms": tok_s * 1e3, "tokenize_bed_text_ms": tok_text_s * 1e3, "ids": int(len(ids)),
            "lines_per_s": n_lines / tok_s, "parity_vs_zlib_and_text_path": all(D.gather_objects(ok)), "data_gen_s": prep_s,
            "note": "gunzip_host_to_host = gtgpu_gunzip from / to host memory (H2D of the members, kernel, D2H of the text); "
                    "tokenize_bed_gz = gz bytes in, token ids out"}


def sub_backend(args, torch, dev, ctx, stream, D, rank, world, peak, universe, offs, s, e, v, other_kind):
    """The headline workload on the OTHER overlapper backend (`tokenizer_type` bits / ailist are both first-class configs,
    gtars-tokenizers/src/config.rs:29-34): same files, device-resident, K steps, parity on a sample of files."""
    from gtars_b200 import ffi, synth
    n_files = max(1, (args.files if args.scaling == "weak" else args.files // world) // 10)   # a tenth of the files
    per_file = args.per_file
    n = n_files * per_file
    t0 = time.perf_counter()
    ix = ffi.Index(ctx, ffi.KIND_AILIST if other_kind == "ailist" else ffi.KIND_BITS, offs, s, e, v)
    build_s = time.perf_counter() - t0
    d_chr = torch.empty(n, dtype=torch.int32, device=dev)
    d_start = torch.empty(n, dtype=torch.int32, device=dev)
    d_end = torch.empty(n, dtype=torch.int32, device=dev)
    chunk = max(1, min(n_files, (32 << 20) // per_file))
    first_file = rank * n_files
    for f0 in range(0, n_files, chunk):
        k = min(chunk, n_files - f0)
        q = synth.make_query_files(universe, k, per_file, device=dev, first_file=first_file + f0, width_scale=args.width_scale)
        sl = slice(f0 * per_file, (f0 + k) * per_file)
        d_chr[sl], d_start[sl], d_end[sl] = q["chr"], q["start"], q["end"]
        del q
    d_fo = torch.arange(n_files + 1, dtype=torch.int64, device=dev) * per_file
    cap = 2 * n + 1024
    d_ids = torch.empty(cap, dtype=torch.int32, device=dev)
    d_tok = torch.empty(n_files + 1, dtype=torch.int64, device=dev)
    d_total = torch.zeros(1, dtype=torch.int64, device=dev)
    step = lambda: ix.find_dev(n, d_chr.data_ptr(), d_start.data_ptr(), d_end.data_ptr(), 0, n_files, d_fo.data_ptr(), d_ids.data_ptr(),
                               cap, None, d_tok.data_ptr(), d_total.data_ptr())
    with torch.cuda.stream(stream):
        for _ in range(3):
            step()
        stream.synchronize()
        hits = int(d_total.item())
        assert hits <= cap
        D.barrier()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record(stream)
        for _ in range(args.steps):
            step()
        ev1.record(stream)
        stream.synchronize()
    ms = D.max(ev0.elapsed_time(ev1) / args.steps)
    # parity: every 10th file, all ids in order
    from oracle import oracle as orc
    files = np.arange(0, n_files, 10)
    g_tok = d_tok.cpu().numpy().astype(np.int64)
    qsel = (torch.from_numpy(files).to(dev).view(-1, 1) * per_file + torch.arange(per_file, device=dev).view(1, -1)).flatten()
    qc, qs, qe = (t[qsel].cpu().numpy().view(np.uint32) for t in (d_chr, d_start, d_end))
    o = orc.Index(orc.AILIST if other_kind == "ailist" else orc.BITS, offs, s, e, v)
    o_off, o_ids = o.tokenize_files((np.arange(len(files) + 1) * per_file).astype(np.uint64), qc, qs, qe, universe["unk_id"], threads=host_threads())
    seg = torch.cat([torch.arange(int(g_tok[f]), int(g_tok[f + 1]), device=dev) for f in files])
    ok = bool(np.array_equal(d_ids[seg].cpu().numpy().view(np.uint32), o_ids))
    info = ix.info()
    algo = 12 * n + 4 * hits + 8 * (n_files + 1) + 12 * info["n_intervals"]
    ix.close()
    return {"workload": f"C2 on the {other_kind} backend: tokenize {n_files} files x {per_file} regions per GPU (a tenth of the headline batch)",
            "backend": other_kind, "queries_per_gpu": n, "ms": ms, "value": D.sum(float(n)) / (ms * 1e-3), "unit": UNIT,
            "algorithmic_bytes": algo, "frac": algo / (ms * 1e-3) / 1e9 / peak, "index_build_s": build_s, "index": info,
            "parity_vs_oracle": all(D.gather_objects(ok)), "parity_files_checked": int(len(files))}


def _fragments(synth, universe, first, k, dev):
    """Fragments [first, first + k) of the C5 stream: nucleosomal width mixture (modes ~50 / 200 / 400 bp), 60 % inside
    peaks, Zipf-ish barcode sizes; unsorted."""
    import torch
    idx = torch.arange(first, first + k, dtype=torch.int64, device=dev)
    seed = synth.SEED_FRAGMENTS
    mode = synth.rand_u63(seed, 1, idx) % 10
    base = torch.where(mode < 4, 50, torch.where(mode < 8, 200, 400))
    width = base + synth.rand_u63(seed, 2, idx) % 60 - 20
    u_chr, u_start, u_end = (universe[x].to(dev).long() for x in ("chr", "start", "end"))
    p = synth.rand_u63(seed, 3, idx) % universe["n"]
    inside = synth.rand_u63(seed, 4, idx) % 10 < 6
    pk_start = torch.clamp(u_start[p] + synth.rand_u63(seed, 5, idx) % torch.clamp(u_end[p] - u_start[p], min=1) - width // 2, min=0)
    bg_chr, bg_start = synth._genome_pos(synth.rand_u63(seed, 6, idx), dev)
    chr_ = torch.where(inside, u_chr[p], bg_chr)
    start = torch.where(inside, pk_start, bg_start)
    csz = torch.tensor(synth.CHROM_SIZES, dtype=torch.int64, device=dev)[chr_]
    start = torch.minimum(start, csz - 1)
    end = torch.minimum(start + width, csz)
    bc = synth.rand_u63(seed, 9, idx) % 100_000
    bc = (bc * bc) // 100_000  # skewed barcode sizes
    return chr_.int(), start.int(), end.int(), bc.int()


# =====================================================================================================================
def main():
    args = parse_args()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    from gtars_b200 import ffi, synth

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    D = Dist(torch, world, dev)
    stream = torch.cuda.Stream(device=dev)
    ctx = ffi.Context(local_rank, stream=stream.cuda_stream)
    kind = ffi.KIND_BITS if args.kind == "bits" else ffi.KIND_AILIST
    peak, peak_src = peaks()
    t_start = time.perf_counter()

    # ---- universe + index (replicated on every rank) ---------------------------------------------------------------
    u = synth.make_universe(args.universe, nested_frac=args.nested, device=dev)
    offs = u["chrom_offsets"].cpu().numpy().astype(np.uint64)
    s, e, v = (u[k].cpu().numpy().view(np.uint32) for k in ("g_start", "g_end", "g_val"))
    t_b = time.perf_counter()
    index = ffi.Index(ctx, kind, offs, s, e, v)
    index_build_s = time.perf_counter() - t_b
    info = index.info()

    # ---- this rank's files, generated on the device (untimed) -------------------------------------------------------
    n_files = args.files if args.scaling == "weak" else args.files // world
    per_file = args.per_file
    n = n_files * per_file
    first_file = rank * n_files
    d_chr = torch.empty(n, dtype=torch.int32, device=dev)
    d_start = torch.empty(n, dtype=torch.int32, device=dev)
    d_end = torch.empty(n, dtype=torch.int32, device=dev)
    chunk = max(1, min(n_files, (32 << 20) // per_file))
    for f0 in range(0, n_files, chunk):
        k = min(chunk, n_files - f0)
        q = synth.make_query_files(u, k, per_file, device=dev, first_file=first_file + f0, width_scale=args.width_scale)
        sl = slice(f0 * per_file, (f0 + k) * per_file)
        d_chr[sl], d_start[sl], d_end[sl] = q["chr"], q["start"], q["end"]
        del q
    d_file_offsets = torch.arange(n_files + 1, dtype=torch.int64, device=dev) * per_file
    cap = n + n // 4 + 1024
    d_ids = torch.empty(cap, dtype=torch.int32, device=dev)
    d_file_tok = torch.empty(n_files + 1, dtype=torch.int64, device=dev)
    d_total = torch.zeros(1, dtype=torch.int64, device=dev)
    torch.cuda.synchronize()

    def step():
        index.find_dev(n, d_chr.data_ptr(), d_start.data_ptr(), d_end.data_ptr(), 0, n_files,
                       d_file_offsets.data_ptr(), d_ids.data_ptr(), cap, None, d_file_tok.data_ptr(),
                       d_total.data_ptr())

    with torch.cuda.stream(stream):
        step()
        stream.synchronize()
        if int(d_total.item()) > cap:  # multi-hit universes (the nested variant): size the id buffer exactly and redo
            cap = int(d_total.item())
            d_ids = torch.empty(cap, dtype=torch.int32, device=dev)
        for _ in range(max(args.warmup, 3)):
            step()
        stream.synchronize()
        hits = int(d_total.item())
        assert hits <= cap, "output capacity too small for the synthetic workload"
        n_empty_files = int((d_file_tok[1:] == d_file_tok[:-1]).sum().item())
        dump = None
        if args.dump_outputs and rank == 0:
            # what a caller of this path receives: the ids of all files and each file's offset into them
            dump = {name: (t, dump_positions(len(t), seed)) for seed, (name, t) in
                    enumerate((("token_ids", d_ids[:hits]), ("file_token_offsets", d_file_tok)))}
            dump_index = {name: torch.from_numpy(pos).to(dev) for name, (_, pos) in dump.items() if pos is not None}

        # ---- timed region: K back-to-back steps, CUDA events on the launching stream ---------------------------------
        sampler = ClockSampler(local_rank)
        launches0 = ctx.launch_count()
        ctx.timing_enable(True)
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        D.barrier()
        torch.cuda.synchronize()
        sampler.start()
        ev0.record(stream)
        for _ in range(args.steps):
            step()
        ev1.record(stream)
        stream.synchronize()
        torch.cuda.synchronize()
        if dump is not None:  # copied before the untimed steps below rewrite the same buffers
            dump = {name: (t[dump_index[name]] if pos is not None else t.clone(), pos) for name, (t, pos) in dump.items()}
        D.barrier()
        kernel_ms = ctx.timing_read()
        ctx.timing_enable(False)
        launches = ctx.launch_count() - launches0
        # K steps of a few ms are shorter than one nvidia-smi sampling period: keep the identical load running (untimed)
        # until the sampler has covered at least half a second, so that the clocks line reflects this workload.
        t_probe = time.perf_counter()
        while time.perf_counter() - t_probe < 0.5:
            for _ in range(8):
                step()
            stream.synchronize()
        clocks = sampler.stop()
        clocks["window"] = "timed region + 0.5 s of the identical steps right behind it"
        ms_per_step = D.max(ev0.elapsed_time(ev1) / args.steps)
        if dump is not None:
            write_dump(args.dump_outputs, {name: (t.cpu().numpy().view(np.uint32) if t.dtype == torch.int32 else t.cpu().numpy(), pos)
                                           for name, (t, pos) in dump.items()})
            del dump, dump_index

    total_queries = D.sum(float(n))
    value = total_queries / (ms_per_step * 1e-3)

    # ---- roofline of the dominant kernel (fused count→scan→emit) ---------------------------------------------------------
    # algorithmic bytes per launch: queries read once (12 B each), ids written once (4 B per hit), per-file offsets
    # written once, index (starts, pmax, vals = 12 B per interval) read once.  Per-query counts/offsets are never
    # materialised, so they are not counted.
    algo_bytes = 12 * n + 4 * hits + 8 * (n_files + 1) + 12 * info["n_intervals"]
    k_ms = statistics.mean(kernel_ms) if kernel_ms else ms_per_step
    achieved = algo_bytes / (k_ms * 1e-3) / 1e9
    traffic, traffic_src = None, None  # dram bytes read + written by this kernel, from the committed ncu --set full capture
    for name in ("r02_traffic.json", "r01_traffic.json"):
        try:
            with open(os.path.join(ROOT, "profiles", name)) as f:
                tr = json.load(f)
            w = tr["workload"]
            if (w["files_per_gpu"], w["regions_per_file"], w["universe_regions"], w["backend"], w["nested_frac"]) == (
                    n_files, args.per_file, args.universe, args.kind, args.nested):
                traffic, traffic_src = tr["dram_bytes_read"] + tr["dram_bytes_write"], f"profiles/{name} (ncu, same command)"
                break
        except Exception:
            pass
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": traffic, "traffic_source": traffic_src,
                "peak_source": peak_src, "kernel": "fused_find_kernel", "kernel_ms": k_ms,
                "algorithmic_bytes_per_launch": algo_bytes, "bytes_per_query": algo_bytes / n,
                "kernel_share_of_step": k_ms / (ev0.elapsed_time(ev1) / args.steps)}

    # ---- full-size parity: >= 10 % of the files, every id and offset, against the multithreaded oracle (untimed) ----------
    parity = None
    try:
        n_chk = min(n_files, max(args.parity_files, 1))
        stride = max(n_files // n_chk, 1)
        files = np.arange(0, n_files, stride)[:n_chk]
        g_tok = d_file_tok.cpu().numpy().astype(np.int64)
        qsel = (torch.from_numpy(files).to(dev).view(-1, 1) * per_file + torch.arange(per_file, device=dev).view(1, -1)).flatten()
        qc, qs, qe = (t[qsel].cpu().numpy().view(np.uint32) for t in (d_chr, d_start, d_end))
        fo_chk = (np.arange(len(files) + 1) * per_file).astype(np.uint64)
        o_off, o_ids = oracle_index(args, u).tokenize_files(fo_chk, qc, qs, qe, u["unk_id"], threads=host_threads())
        seg = torch.cat([torch.arange(int(g_tok[f]), int(g_tok[f + 1]), device=dev) for f in files]) if len(files) else None
        g_ids = d_ids[seg].cpu().numpy().view(np.uint32)
        g_len = (g_tok[files + 1] - g_tok[files])
        # raw device offsets carry no [unk] insertions: a file without a hit has an empty run there and [unk] in the oracle
        o_len = np.diff(o_off.astype(np.int64))
        same_len = bool(np.array_equal(np.where(g_len == 0, 1, g_len), o_len))
        same_ids = bool(n_empty_files > 0 or np.array_equal(g_ids, o_ids))
        ok = same_len and same_ids
        parity = {"files_checked": int(len(files)), "queries_checked": int(len(qc)), "ids_checked": int(len(g_ids)),
                  "equal_to_oracle": ok, "digest_gpu": digest64(g_len, g_ids), "digest_oracle": digest64(o_len, o_ids),
                  "oracle_threads": host_threads(), "what": f"every {stride}th file of this rank's {n_files}: all ids in order + per-file id counts"}
        del qsel, seg
    except Exception as ex:  # never lose the headline to the checker
        parity = {"error": repr(ex)}
    parity_ok = all(bool(p and p.get("equal_to_oracle")) for p in D.gather_objects(parity))

    # ---- e2e: the C-ABI host entry point with pinned host buffers --------------------------------------------------------
    e2e = None
    pcie = None
    if not args.no_e2e:
        # What a Rust caller holds after RegionSet::try_from + a chromosome-name lookup: flat (chr id, start, end) arrays.
        # A host-side packer (multithreaded C++) turns them into a wire format of the host entry point:
        #   packed  (default) gtgpu_marshal_packed -> gtgpu_tokenize_files_packed: chromosome runs, ONE u32 per region (offset from
        #           the anchor of its 32-region block | width) + the anchors + an exception list: 4.125 B of PCIe per region;
        #   compact gtgpu_marshal_compact -> gtgpu_tokenize_files_compact: runs, u32 starts, u16 widths: 6 B per region;
        #   runs    runs + u32 starts + u32 ends: 8 B per region (instead of the 12 B of the flat arrays).
        api = args.e2e_api
        packed, compact = api == "packed", api == "compact"
        h_chr = np.empty(n, dtype=np.uint32)
        h_start = ffi.pinned_empty(n, np.uint32) if not packed else np.empty(n, dtype=np.uint32)
        h_end = ffi.pinned_empty(n, np.uint32) if api == "runs" else np.empty(n, dtype=np.uint32)
        torch.from_numpy(h_chr.view(np.int32)).copy_(d_chr)
        torch.from_numpy(h_start.view(np.int32)).copy_(d_start)
        torch.from_numpy(h_end.view(np.int32)).copy_(d_end)
        h_fo = d_file_offsets.cpu().numpy().astype(np.uint64)
        h_w16 = ffi.pinned_empty(n, np.uint16) if not packed else None
        h_pk = ffi.pinned_empty(n, np.uint32) if packed else None
        h_an = ffi.pinned_empty((n + 31) // 32, np.uint32) if packed else None
        marshal_s = []
        for _ in range(2):
            t0 = time.perf_counter()
            if packed:
                h_run_off, h_run_chr, pk_bits, _, _, h_exc_idx, h_exc_start, h_exc_end = ffi.marshal_packed(
                    h_chr, h_start, h_end, h_fo, packed_out=h_pk, anchors_out=h_an)
            else:
                h_run_off, h_run_chr, _, h_wide_idx, h_wide_end = ffi.marshal_compact(h_chr, h_start, h_end, h_fo, width16_out=h_w16)
            marshal_s.append(time.perf_counter() - t0)
        marshal_s = D.max(min(marshal_s))
        del h_chr
        if api != "runs":
            del h_end
        if packed:
            del h_start
        torch.cuda.synchronize()
        L = ffi.lib()

        def e2e_on(ix):
            if packed:
                return ix.tokenize_files_packed(h_fo, h_run_off, h_run_chr, pk_bits, h_pk, h_an, h_exc_idx, h_exc_start, h_exc_end,
                                                u["unk_id"], keep_buf=True)
            if compact:
                return ix.tokenize_files_compact(h_fo, h_run_off, h_run_chr, h_start, h_w16, h_wide_idx, h_wide_end, u["unk_id"],
                                                 keep_buf=True)
            return ix.tokenize_files_runs(h_fo, h_run_off, h_run_chr, h_start, h_end, u["unk_id"], keep_buf=True)

        def e2e_call():
            return e2e_on(index)

        def e2e_step():
            off, buf = e2e_call()
            total = int(off[-1])  # the step's result is read on the host
            assert L.gtgpu_buf_len(buf) == total
            L.gtgpu_buf_free(buf)
            return total

        # the host entry point must return exactly what the device-resident path produced
        off_chk, buf_chk = e2e_call()
        k_chk = min(int(off_chk[-1]), 4_000_000)
        ids_chk = np.ctypeslib.as_array(C.cast(L.gtgpu_buf_data(buf_chk), C.POINTER(C.c_uint32)), shape=(int(off_chk[-1]),))
        e2e_matches_device = bool(n_empty_files > 0 or (np.array_equal(ids_chk[:k_chk], d_ids[:k_chk].cpu().numpy().view(np.uint32))
                                                        and np.array_equal(ids_chk[-k_chk:], d_ids[hits - k_chk:hits].cpu().numpy().view(np.uint32))))
        del ids_chk
        L.gtgpu_buf_free(buf_chk)

        for _ in range(2):
            e2e_total = e2e_step()
        D.barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            e2e_step()
        torch.cuda.synchronize()
        D.barrier()
        e2e_s = D.max((time.perf_counter() - t0) / args.steps)
        if packed:
            h2d_q = 4 * n + 4 * ((n + 31) // 32) + 16 * len(h_exc_idx)
        elif compact:
            h2d_q = 6 * n + 12 * len(h_wide_idx)
        else:
            h2d_q = 8 * n
        h2d = h2d_q + 8 * (n_files + 1) + 12 * len(h_run_chr) + 8
        d2h = 4 * e2e_total + 8 * (n_files + 1)
        api_text = {
            "packed": "gtgpu_tokenize_files_packed (pinned host: one u32 per region = offset from its 32-region block anchor | width, "
                      "+ anchors + exceptions + chromosome runs in, pinned result buffer out)",
            "compact": "gtgpu_tokenize_files_compact (pinned host start u32 + width u16 + chromosome runs in, pinned result buffer out)",
            "runs": "gtgpu_tokenize_files_runs (pinned host start/end + chromosome runs in, pinned result buffer out)"}[api]
        e2e = {"value": total_queries / e2e_s, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
               "ms_per_step": e2e_s * 1e3, "api": api_text,
               "ids_match_device_resident_path": e2e_matches_device, "chromosome_runs": int(len(h_run_chr)),
               "marshal": {"seconds": marshal_s, "threads": host_threads(),
                           "what": ("gtgpu_marshal_packed" if packed else "gtgpu_marshal_compact") + ": flat (chr id, start, end) u32 "
                                   "arrays -> the wire format above, host side, NOT inside ms_per_step",
                           "value_with_marshal": total_queries / (e2e_s + marshal_s), "unit": UNIT}}
        if packed:
            e2e["packed"] = {"width_bits": int(pk_bits), "exceptions": int(len(h_exc_idx)), "bytes_per_region": h2d_q / max(n, 1)}
        assert e2e_total == hits + n_empty_files
        if world > 1:
            # The drop-in form of multi-GPU use: ONE process (rank 0) drives all N GPUs through a multi-device context
            # (gtgpu_init_multi) and the same entry point; its 1e9 queries are dealt to the devices chunk by chunk (strong
            # scaling of one caller's batch).  The other ranks wait on the host meanwhile, their GPUs idle.
            torch.cuda.synchronize()
            D.barrier()
            try:
                if rank == 0:
                    mctx = ffi.Context(devices=list(range(world)))
                    mindex = ffi.Index(mctx, kind, offs, s, e, v)

                    def m_call():
                        return e2e_on(mindex)
                    off_m, buf_m = m_call()
                    ids_m = np.ctypeslib.as_array(C.cast(L.gtgpu_buf_data(buf_m), C.POINTER(C.c_uint32)), shape=(int(off_m[-1]),))
                    same = bool(int(off_m[-1]) == e2e_total and (n_empty_files > 0 or (
                        np.array_equal(ids_m[:k_chk], d_ids[:k_chk].cpu().numpy().view(np.uint32))
                        and np.array_equal(ids_m[-k_chk:], d_ids[hits - k_chk:hits].cpu().numpy().view(np.uint32)))))
                    del ids_m
                    L.gtgpu_buf_free(buf_m)
                    t0 = time.perf_counter()
                    for _ in range(args.steps):
                        off_m, buf_m = m_call()
                        L.gtgpu_buf_free(buf_m)
                    m_s = (time.perf_counter() - t0) / args.steps
                    e2e["single_process_multi_device"] = {
                        "devices": world, "queries": n, "ms_per_call": m_s * 1e3, "value": n / m_s, "unit": UNIT,
                        "ids_match_device_resident_path": same, "scaling": "strong (one caller's batch over all devices)",
                        "api": f"gtgpu_init_multi + gtgpu_tokenize_files_{api}: chunks dealt round-robin to the devices, ids land "
                               "at their final offsets in one pinned buffer"}
                    mindex.close()
                    mctx.close()
            except Exception as ex:
                e2e["single_process_multi_device"] = {"error": repr(ex)}
            D.host_barrier()
        for h_buf in ([h_pk, h_an] if packed else [h_start, h_w16] + ([h_end] if api == "runs" else [])):
            ffi.pinned_free(h_buf)
        if not args.no_pcie_probe:
            try:
                pcie = pcie_probe(torch, dev, D, h2d, d2h)
                e2e["pcie_floor_ms"] = pcie["floor_ms_for_one_e2e_step"]
                e2e["frac_of_pcie_ceiling"] = pcie["floor_ms_for_one_e2e_step"] / (e2e_s * 1e3)
            except Exception as ex:
                pcie = {"error": repr(ex)}

    # ---- cpu baseline (rank 0, N = 1) ------------------------------------------------------------------------------------
    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu:
        u_cpu = {k: (t.cpu() if hasattr(t, "cpu") else t) for k, t in u.items()}
        rate, sample = cpu_oracle_rate(args, 1, args.cpu_seconds, u_cpu)
        cpu_baseline = {"value": rate, "unit": UNIT, "cores": 1, "kind": "port", "sample": sample,
                        "note": "C++ restatement of gtars' algorithm (the Rust reference cannot be built here); 1 thread because "
                                "the reference path is single-threaded.  It returns ids directly and so omits the reference's "
                                "per-hit id -> String -> id round trip (tokenizer.rs:146-171): real gtars is slower than this"}
    c2_seconds = time.perf_counter() - t_start

    # ---- sub-records: the other BASELINE configs, sharded over the ranks ---------------------------------------------------
    del d_chr, d_start, d_end, d_ids
    torch.cuda.empty_cache()
    configs = {}
    wanted = [c for c in args.configs.split(",") if c]
    for name in wanted:
        t0 = time.perf_counter()
        try:
            if name == "c3":
                rec = sub_c3(args, torch, dev, ctx, stream, D, rank, world, peak)
            elif name == "c4":
                rec = sub_c4(args, torch, dev, ctx, stream, D, rank, world, peak)
            elif name == "c5":
                rec = sub_c5(args, torch, dev, ctx, stream, D, rank, world, peak, u, index)
            elif name == "gz":
                rec = sub_gz(args, torch, dev, ctx, stream, D, rank, world, peak, u, index)
            elif name == "backend":
                rec = sub_backend(args, torch, dev, ctx, stream, D, rank, world, peak, u, offs, s, e, v,
                                  "ailist" if args.kind == "bits" else "bits")
            else:
                continue
        except Exception as ex:
            rec = {"error": repr(ex), "trace": traceback.format_exc()[-1500:]}
        rec["seconds_in_bench"] = time.perf_counter() - t0
        configs[name] = rec
        torch.cuda.empty_cache()

    if rank == 0:
        details = {"hits_per_gpu": hits, "index": info, "index_build_s": index_build_s, "c2_seconds": c2_seconds,
                   "host_threads": host_threads(), "empty_files": n_empty_files}
        out = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "u32",
            "data": "synthetic", "config": workload_config(args, world), "roofline": roofline, "cpu_baseline": cpu_baseline,
            "e2e": e2e, "gpu_launches": launches, "clocks": clocks, "parity": parity, "parity_all_ranks": parity_ok,
            "pcie": pcie, "details": details, "configs": configs,
        }
        print(json.dumps(out))
    index.close()
    ctx.close()
    D.close()


if __name__ == "__main__":
    main()
