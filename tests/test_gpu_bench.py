"""bench.py on the device: --steps sets the timed steps, and --dump-outputs writes the headline path's result of the last
timed step, which must equal the CPU oracle on the same seeded inputs."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dump_outputs_equal_oracle(tmp_path):
    from gtars_b200 import synth
    from oracle import oracle as orc
    files, per_file, universe = 20, 5000, 20_000
    out = tmp_path / "dump"
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--files", str(files), "--per-file", str(per_file),
           "--universe", str(universe), "--steps", "3", "--warmup", "1", "--no-e2e", "--no-cpu", "--no-pcie-probe",
           "--configs", "", "--dump-outputs", str(out)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["steps"] == 3 and line["parity"]["equal_to_oracle"] and line["details"]["empty_files"] == 0
    assert sorted(os.listdir(out)) == ["file_token_offsets.npy", "token_ids.npy"]   # small enough: no sampling
    offs, ids = np.load(out / "file_token_offsets.npy"), np.load(out / "token_ids.npy")
    assert offs.dtype == np.float64 and ids.dtype == np.float64
    u = synth.make_universe(universe)
    q = synth.make_query_files(u, files, per_file)
    o = orc.Index(orc.BITS, u["chrom_offsets"].numpy().astype(np.uint64),
                  *(u[k].numpy().view(np.uint32) for k in ("g_start", "g_end", "g_val")))
    o_off, o_ids = o.tokenize_files(q["file_offsets"].numpy().astype(np.uint64),
                                    *(q[k].numpy().view(np.uint32) for k in ("chr", "start", "end")), u["unk_id"])
    assert np.array_equal(offs, o_off.astype(np.float64)) and np.array_equal(ids, o_ids.astype(np.float64))
    assert len(ids) == line["details"]["hits_per_gpu"]
