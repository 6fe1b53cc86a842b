"""Host-only checks of bench.py (no GPU): the reference arm, the config both arms share, helpers."""
import importlib.util
import json
import os
import subprocess
import sys
import types

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench():
    spec = importlib.util.spec_from_file_location("bench_under_test", os.path.join(ROOT, "bench.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def test_reference_arm_uses_all_host_threads_even_under_torchrun_env():
    """torch.distributed.run exports OMP_NUM_THREADS=1; the reference arm must still use every CPU it may run on, the same
    bounded sample at every N, and print the config our arm prints (so the driver's same_config check holds)."""
    env = dict(os.environ, OMP_NUM_THREADS="1", RANK="0", WORLD_SIZE="4", LOCAL_RANK="0")
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "4", "--files", "6", "--per-file", "3000",
           "--universe", "20000", "--steps", "1", "--warmup", "1"]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=300, env=env, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["n_gpus"] == 4
    assert line["cpu_baseline"]["cores"] == len(os.sched_getaffinity(0))
    assert line["cpu_baseline"]["kind"] == "port" and line["value"] > 0 and line["e2e"]["value"] == line["value"]
    b = _bench()
    args = types.SimpleNamespace(files=6, per_file=3000, universe=20000, kind="bits", nested=0.0, width_scale=1, scaling="weak")
    assert line["config"] == b.workload_config(args, 4)
    # other ranks print nothing and exit 0
    env["RANK"] = "2"
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=300, env=env, cwd=ROOT)
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_workload_config_carries_no_diagnostics_and_strong_scaling_divides_files():
    b = _bench()
    args = types.SimpleNamespace(files=10_000, per_file=100_000, universe=1_000_000, kind="bits", nested=0.0, width_scale=1, scaling="weak")
    weak = b.workload_config(args, 8)
    assert weak["files_per_gpu"] == 10_000 and weak["scaling"] == "weak"
    assert not any(k.startswith("parity") or k in ("hits_per_gpu", "index") for k in weak)
    args.scaling = "strong"
    assert b.workload_config(args, 8)["files_per_gpu"] == 1250


def test_host_threads_ignores_omp_num_threads(monkeypatch):
    b = _bench()
    monkeypatch.setenv("OMP_NUM_THREADS", "1")
    assert b.host_threads() == len(os.sched_getaffinity(0))
    from oracle import oracle as orc
    assert orc.max_threads() == len(os.sched_getaffinity(0))


def test_digest_is_order_sensitive():
    b = _bench()
    a = np.arange(10, dtype=np.uint32)
    assert b.digest64(a) == b.digest64(a.copy())
    assert b.digest64(a) != b.digest64(a[::-1])
    assert b.digest64(a[:5], a[5:]) == b.digest64(a)


def test_dump_outputs_sample_is_fixed_bounded_and_float64(tmp_path):
    b = _bench()
    assert b.dump_positions(b.DUMP_MAX_VALUES, 0) is None
    n = 1_000_000_000
    p = b.dump_positions(n, 0)
    assert len(p) == b.DUMP_MAX_VALUES and np.all(np.diff(p) > 0) and p[0] >= 0 and p[-1] < n
    assert np.array_equal(p, b.dump_positions(n, 0)) and not np.array_equal(p, b.dump_positions(n, 1))
    ids = np.array([0, 7, 0xFFFFFFFF], dtype=np.uint32)
    b.write_dump(str(tmp_path / "d"), {"ids": (ids, None), "offs": (np.arange(5, dtype=np.int64), np.array([0, 2, 9]))})
    got = {f: np.load(tmp_path / "d" / f) for f in sorted(os.listdir(tmp_path / "d"))}
    assert sorted(got) == ["ids.npy", "offs.npy", "offs_positions.npy"] and all(a.dtype == np.float64 for a in got.values())
    assert got["ids.npy"].tolist() == [0, 7, 0xFFFFFFFF] and got["offs_positions.npy"].tolist() == [0, 2, 9]
    # four arrays at the cap (ids, offsets and their positions) stay within 64 MB
    assert 4 * (8 * b.DUMP_MAX_VALUES + 128) <= 64 << 20


def test_steps_must_be_positive():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "0"],
                       capture_output=True, text=True, timeout=120, cwd=ROOT)
    assert r.returncode == 2 and "--steps" in r.stderr


def test_marshal_compact_matches_numpy():
    """gtgpu_marshal_compact is host code: runs cut at chromosome changes and file boundaries, u16 widths, exceptions."""
    from gtars_b200 import ffi
    rng = np.random.default_rng(7)
    n = 2_500_000
    fo = np.array([0, 10, 10, 1_200_000, n], dtype=np.uint64)
    chr_ = np.sort(rng.integers(0, 5, n)).astype(np.uint32)
    start = rng.integers(0, 1 << 30, n).astype(np.uint32)
    end = (start + rng.integers(0, 70000, n)).astype(np.uint32)
    end[5] = start[5] - 3
    for threads in (1, 3, 0):
        ro, rc, w16, wi, we = ffi.marshal_compact(chr_, start, end, fo, threads=threads)
        cut = np.zeros(n, bool)
        cut[0] = True
        cut[1:] = chr_[1:] != chr_[:-1]
        cut[fo[fo < n].astype(np.int64)] = True
        exp = np.flatnonzero(cut)
        assert np.array_equal(ro[:-1], exp) and ro[-1] == n and np.array_equal(rc, chr_[exp])
        wide = (end < start) | ((end.astype(np.int64) - start) > 0xFFFE)
        assert np.array_equal(wi, np.flatnonzero(wide)) and np.array_equal(we, end[wide])
        assert np.array_equal(w16[~wide], (end - start)[~wide].astype(np.uint16)) and (w16[wide] == 0xFFFF).all()
    ro, rc, w16, wi, we = ffi.marshal_compact(chr_[:0], start[:0], end[:0], np.zeros(1, np.uint64))
    assert len(rc) == 0 and len(wi) == 0 and ro[0] == 0


def _unpack(n, wb, pk, an, xi, xs, xe):
    off_bits = 32 - wb
    start = (an[np.arange(n) >> 5] + (pk & np.uint32((1 << off_bits) - 1))).astype(np.uint32)
    end = (start + (pk >> np.uint32(off_bits))).astype(np.uint32)
    start[xi.astype(np.int64)] = xs
    end[xi.astype(np.int64)] = xe
    return start, end


def test_marshal_packed_round_trips():
    """gtgpu_marshal_packed is host code: whatever the input, (packed, anchors, exceptions) decode to the caller's arrays; sorted
    files cost few exceptions (only around run boundaries), unsorted input degrades to exceptions but stays exact."""
    from gtars_b200 import ffi
    rng = np.random.default_rng(11)
    n_files, per = 7, 150_001                       # odd sizes: file and run boundaries fall inside 32-query blocks
    n = n_files * per
    fo = (np.arange(n_files + 1) * per).astype(np.uint64)
    chr_ = np.concatenate([np.sort(rng.integers(0, 25, per)) for _ in range(n_files)]).astype(np.uint32)
    start = rng.integers(0, 200_000_000, n).astype(np.uint32)
    # RegionSet::sort order inside every file: by chromosome, then start
    for f in range(n_files):
        a, b = f * per, (f + 1) * per
        o = np.lexsort((start[a:b], chr_[a:b]))
        start[a:b] = start[a:b][o]
    end = (start + rng.integers(150, 1000, n)).astype(np.uint32)
    end[5] = start[5] - 3                            # reversed
    end[77_777] = start[77_777] + 5_000_000          # wide
    for threads in (1, 3, 0):
        ro, rc, wb, pk, an, xi, xs, xe = ffi.marshal_packed(chr_, start, end, fo, threads=threads)
        ro2, rc2, _, _, _ = ffi.marshal_compact(chr_, start, end, fo, threads=threads)
        assert np.array_equal(ro, ro2) and np.array_equal(rc, rc2)
        assert 6 <= wb <= 16 and len(an) == (n + 31) // 32
        assert np.all(np.diff(xi.astype(np.int64)) > 0) and {5, 77_777} <= set(xi.tolist())
        assert len(xi) < 32 * len(rc)                # only blocks that hold a run boundary have exceptions (+ the two above)
        s2, e2 = _unpack(n, wb, pk, an, xi, xs, xe)
        assert np.array_equal(s2, start) and np.array_equal(e2, end)
    # a fixed split, unsorted starts, a ragged tail block
    m = 100_003
    us, ue = rng.integers(0, 1 << 32, m, dtype=np.uint64).astype(np.uint32), rng.integers(0, 1 << 32, m, dtype=np.uint64).astype(np.uint32)
    ro, rc, wb, pk, an, xi, xs, xe = ffi.marshal_packed(chr_[:m], us, ue, np.array([0, m], np.uint64), width_bits=12)
    assert wb == 12
    s2, e2 = _unpack(m, wb, pk, an, xi, xs, xe)
    assert np.array_equal(s2, us) and np.array_equal(e2, ue)
    ro, rc, wb, pk, an, xi, xs, xe = ffi.marshal_packed(chr_[:0], start[:0], end[:0], np.zeros(1, np.uint64))
    assert len(rc) == 0 and len(xi) == 0 and ro[0] == 0
