"""Result buffers (gtgpu_buf) across failed calls and threads: a failed BGZF fragment call whose text copy was in flight
leaves the context usable, and results are freed from another thread while a call runs on the same context."""
import re
import threading

import numpy as np
import pytest

from tests.test_gpu_inflate import bgzf

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    from gtars_b200 import ffi
    c = ffi.Context(0)
    yield c
    c.close()


@pytest.fixture(scope="module")
def universe():
    from gtars_b200 import synth
    return synth.make_universe(200_000)


@pytest.fixture(scope="module")
def index(ctx, universe):
    from gtars_b200 import ffi
    offs = universe["chrom_offsets"].numpy().astype(np.uint64)
    s, e, v = (universe[k].numpy().view(np.uint32) for k in ("g_start", "g_end", "g_val"))
    ix = ffi.Index(ctx, ffi.KIND_BITS, offs, s, e, v)
    yield ix
    ix.close()


def test_failed_gz_fragment_call_then_a_good_one(index, universe):
    """tokenize_fragments_gz fails on a malformed line after the inflated text's copy to the host was enqueued: the error is
    the text form's, and the next call on the same context returns what the text form returns."""
    from gtars_b200 import ffi, synth
    names, unk = list(synth.CHROM_NAMES), int(universe["unk_id"])
    good = synth.fragment_text(*synth.make_fragment_arrays(400_000, 5, 3_000)).tobytes()
    line = len(good) // synth.FRAGMENT_LINE * 3 // 4
    bad = bytearray(good)
    bad[line * synth.FRAGMENT_LINE + 6] = ord("x")                        # the start field of one line is no longer a number
    bad = bytes(bad)

    with pytest.raises(ffi.GtarsGpuError) as want:
        index.tokenize_fragments_text(bad, names, unk)
    bad_gz = bgzf(bad)
    with pytest.raises(ffi.GtarsGpuError) as got:
        index.tokenize_fragments_text(bad_gz, names, unk, gz_member_offsets=ffi.gzip_members(bad_gz))
    assert want.value.code == got.value.code == 1
    at = [re.search(r"at line: (\d+)", str(e.value)).group(1) for e in (want, got)]
    assert at[0] == at[1]

    good_gz = bgzf(good)
    b_gz, o_gz, i_gz = index.tokenize_fragments_text(good_gz, names, unk, gz_member_offsets=ffi.gzip_members(good_gz))
    b_txt, o_txt, i_txt = index.tokenize_fragments_text(good, names, unk)
    assert len(b_txt) > 1000
    assert b_gz == b_txt and np.array_equal(o_gz, o_txt) and np.array_equal(i_gz, i_txt)


def test_free_from_another_thread_during_a_call(index, universe):
    """gtgpu_buf_free from a second thread while tokenize_files runs on the same context (ctypes drops the GIL for both):
    both complete and the call returns what it returns alone."""
    from gtars_b200 import ffi, synth
    q = synth.make_query_files(universe, 16, 500_000, unknown_frac_ppm=1000)
    fo = q["file_offsets"].numpy().astype(np.uint64)
    qc, qs, qe = (q[k].numpy().view(np.uint32) for k in ("chr", "start", "end"))
    unk = int(universe["unk_id"])
    want_off, want_ids = index.tokenize_files(fo, qc, qs, qe, unk)

    small = synth.make_query_files(universe, 4, 20_000, seed=11)
    sfo = small["file_offsets"].numpy().astype(np.uint64)
    sc, ss, se = (small[k].numpy().view(np.uint32) for k in ("chr", "start", "end"))
    held = [index.tokenize_files(sfo[:k + 2], sc, ss, se, unk, keep_buf=True)[1] for k in range(3)]
    held += [index.tokenize_files(sfo, sc, ss, se, unk, keep_buf=True)[1] for _ in range(3)]

    start = threading.Barrier(2)
    status = []

    def free_all():
        start.wait()
        status.extend(ffi.lib().gtgpu_buf_free(h) for h in held)

    t = threading.Thread(target=free_all)
    t.start()
    start.wait()
    got_off, got_ids = index.tokenize_files(fo, qc, qs, qe, unk)
    t.join()
    assert status == [0] * len(held)
    assert np.array_equal(got_off, want_off) and np.array_equal(got_ids, want_ids)
