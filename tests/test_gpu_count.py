"""The counting path called through every entry point: gtgpu_count, gtgpu_any, gtgpu_bits_count and gtgpu_count_dev.

Counting runs on five kernels (kernels.cu): count_kernel (one query per thread, arrays that are not 16-byte aligned),
count_kernel_x4 (four queries per thread, a prefetch of the next step and a tail for n % 4), and the bucketed pass
count_stage_kernel -> count_runs_kernel -> count_unstage_kernel for rank LUTs beyond the L2.  Every search reads one 64-bit
rank-LUT word (index.cu): a base index, a 3-bit count and up to rank_inline = min(4, 29 / rank_shift) in-bin offsets; a count
of 7 marks a crowded bin, which is bisected (the bucketed pass first finds its chromosome with rank_lin_bisect).

Every output element is compared with oracle.Index.  The helpers below restate, from the inputs and the knobs, what the library
will choose (rank shift, words per chromosome, whether rank_lin exists, bucketed or direct, the bucket plan), and every call
asserts through ctx.launch_count() that it ran the path it was meant to reach: 3 launches for the bucketed pass, 1 for a direct
one.  Device outputs start out filled with sentinels between guard bands, so a missing or stray write shows.
"""
import os
import types

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

U32 = 0xFFFFFFFF
SENT32 = 0xA5A5A5A5
GUARD = 64              # sentinel words before and after every device output
HUGE_BINS = str(1 << 40)  # GTGPU_RANK_BINS_PER_INTERVAL that leaves the base rank shift at 0 for every index here
BITS, AILIST = 0, 1

# kernels.cu geometry
CP_TILE = 4096          # queries per tile of the bucketed pass
CP_MAX_BUCKETS = 256
CR_MINBLOCKS = 4        # GT_CR_MINBLOCKS
CR_RUNS = 4
X4_STRIDE_BLOCKS = 32   # direct grids: at most 32 blocks of 256 threads per SM


# ---- a Python statement of the plan ---------------------------------------------------------------------------------------
def rank_inline(sigma):
    return 4 if sigma == 0 else min(4, 29 // sigma)


def _maxima(offs, a):
    return np.array([int(a[lo:hi].max()) if hi > lo else 0 for lo, hi in zip(offs[:-1].astype(np.int64), offs[1:].astype(np.int64))],
                    np.int64)


def rank_plan(offs, s, e):
    """What gtgpu_index_build makes of the rank LUTs (index.cu) under the knobs set now: the shift, rank_inline, the words of
    each chromosome in the starts and the ends block (nb bins + one sentinel, nb = 0 for an empty chromosome), and whether the
    linearised keys of the bucketed pass (rank_lin) fit 32 bits."""
    offs = np.asarray(offs, np.uint64)
    s, e = np.asarray(s, np.uint32), np.asarray(e, np.uint32)
    total = len(s)
    lens = np.diff(offs.astype(np.int64))
    mcs, mce = _maxima(offs, s), _maxima(offs, e)  # the last element of each chromosome's sorted starts / ends

    def entries(m, sh):
        return int(((m >> sh) + 2).sum())

    bpi = os.environ.get("GTGPU_RANK_BINS_PER_INTERVAL")
    budget = max(total, 4096) if bpi is None else max(int(bpi) * total, 4096)
    sigma = 0
    while sigma < 29 and max(entries(mcs, sigma), entries(mce, sigma)) > budget:
        sigma += 1
    extra = os.environ.get("GTGPU_RANK_SHIFT_EXTRA")
    if extra is not None:
        sigma = min(29, sigma + max(0, int(extra)))
    nb_cs = np.where(lens > 0, (mcs >> sigma) + 1, 0)
    nb_ce = np.where(lens > 0, (mce >> sigma) + 1, 0)
    lut_cs = np.concatenate([[0], np.cumsum(nb_cs + 1)])[:-1]
    words_s = int((nb_cs + 1).sum())
    words_e = int((nb_ce + 1).sum())
    return types.SimpleNamespace(
        sigma=sigma, inline=rank_inline(sigma), nb_cs=nb_cs, nb_ce=nb_ce, lut_cs=lut_cs, words_s=words_s, words_e=words_e,
        lut_len=words_s + words_e, has_lin=(words_s << sigma) <= U32 and (words_e << sigma) <= U32,
        proper=bool((s <= e).all()), n_chroms=len(offs) - 1)


def wants_partition(plan, n, min_overlap=0, aligned_in=True):
    """count_wants_partition: whether a call of n queries goes through the bucketed pass."""
    if min_overlap > 1 or not plan.proper or n >= 1 << 31 or plan.lut_len == 0 or not plan.has_lin:
        return False
    if not aligned_in:
        return False
    force = os.environ.get("GTGPU_COUNT_PARTITION")
    if force is not None:
        return force[:1] == "1"
    return plan.lut_len * 8 > (64 << 20) and n >= 4 << 20


def path(plan, n, min_overlap=0, aligned_in=True, aligned_out=True):
    """The kernels a call runs: None (n == 0), "bucketed", "x4" or "scalar"."""
    if n == 0:
        return None
    if wants_partition(plan, n, min_overlap, aligned_in):
        return "bucketed"
    return "x4" if aligned_in and aligned_out else "scalar"


LAUNCHES = {None: 0, "bucketed": 3, "x4": 1, "scalar": 1}


def bucket_plan(plan, n, sm_count):
    """launch_count_bucketed_mode: (bucket count, bucket_shift)."""
    lut_bytes = plan.lut_len * 8
    held = sm_count * CR_MINBLOCKS * 8 * 2 * CR_RUNS * CP_TILE
    nb = 32
    while nb < 128 and (lut_bytes // nb > 16 << 20 or (held // nb) * float(lut_bytes) / float(n) > float(64 << 20)):
        nb *= 2
    force = os.environ.get("GTGPU_COUNT_BUCKETS")
    if force is not None:
        nb = min(CP_MAX_BUCKETS, max(2, int(force)))
    shift = 0
    while (plan.words_s >> shift) >= nb:
        shift += 1
    return nb, shift


def bucket_of(plan, nb, shift, c, e):
    """The bucket count_stage_kernel puts a staged query (c, *, e) in: the starts-LUT word of its end key."""
    key = (int(plan.lut_cs[c]) << plan.sigma) + min(int(e), int(plan.nb_cs[c]) << plan.sigma)
    return min((key >> plan.sigma) >> shift, nb - 1)


# ---- harness ---------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def env():
    """One context on a torch stream: every fill, copy and library call of this module is ordered on that stream."""
    import torch
    from gtars_b200 import ffi
    stream = torch.cuda.Stream()
    ctx = ffi.Context(0, stream=stream.cuda_stream)
    sm = torch.cuda.get_device_properties(0).multi_processor_count
    yield types.SimpleNamespace(ctx=ctx, stream=stream, sm=sm)
    stream.synchronize()
    ctx.close()


def build(env, kind, offs, s, e):
    """(device index, oracle index, plan) over chromosome-grouped arrays, under the knobs set now."""
    from gtars_b200 import ffi
    from oracle import oracle as orc
    offs = np.asarray(offs, np.uint64)
    ix = ffi.Index(env.ctx, kind, offs, s, e)
    return ix, orc.Index(kind, offs, s, e), rank_plan(offs, s, e)


def assert_same(got, want, what):
    got, want = np.asarray(got), np.asarray(want)
    assert got.shape == want.shape, f"{what}: {got.shape} != {want.shape}"
    bad = np.flatnonzero(got != want)
    assert len(bad) == 0, f"{what}: {len(bad)} of {len(want)} differ, first at {bad[0]}: got {int(got[bad[0]])}, want {int(want[bad[0]])}"


def launched(env, fn):
    n0 = env.ctx.launch_count()
    r = fn()
    return r, env.ctx.launch_count() - n0


def check_host(env, ix, o, plan, q, m=0, what=""):
    """count, any and (Bits) bits_count through the host entry points, each on the path the plan names, against the oracle.
    Returns the oracle's counts."""
    from oracle import oracle as orc
    qc, qs, qe = q
    n = len(qc)
    p = path(plan, n, m)
    want = o.count(qc, qs, qe, m, threads=orc.max_threads())
    got, k = launched(env, lambda: ix.count(qc, qs, qe, m))
    assert k == LAUNCHES[p], f"{what}: count ran {k} launches, the {p} path is {LAUNCHES[p]}"
    assert_same(got, want, f"{what}: count ({p}, min_overlap {m})")
    got, k = launched(env, lambda: ix.any(qc, qs, qe, m))
    assert k == LAUNCHES[p], f"{what}: any ran {k} launches, the {p} path is {LAUNCHES[p]}"
    assert_same(got, o.any(qc, qs, qe, m) if n <= 1 << 20 else want > 0, f"{what}: any ({p}, min_overlap {m})")
    if ix.kind == BITS:
        p0 = path(plan, n)
        got, k = launched(env, lambda: ix.bits_count(qc, qs, qe))
        assert k == LAUNCHES[p0], f"{what}: bits_count ran {k} launches, the {p0} path is {LAUNCHES[p0]}"
        assert_same(got, o.bits_count(qc, qs, qe, threads=orc.max_threads()), f"{what}: bits_count ({p0})")
    return want


def run_count_dev(env, ix, q, m=0, offsets=(0, 0, 0, 0)):
    """gtgpu_count_dev with chr / start / end / out placed `offsets` elements past 16-byte aligned bases; the output lies
    between GUARD sentinel words on either side.  Returns (counts, launches); asserts the guard bands are untouched."""
    import torch
    qc, qs, qe = q
    n = len(qc)
    oc, os_, oe, oo = offsets
    with torch.cuda.stream(env.stream):
        bases = [torch.empty(n + 4, dtype=torch.int32, device="cuda") for _ in range(3)]  # 512-byte aligned blocks
        ptrs = []
        for base, a, off in zip(bases, q, (oc, os_, oe)):
            assert base.data_ptr() % 16 == 0
            if n:
                base[off:off + n].copy_(torch.from_numpy(np.ascontiguousarray(a, np.uint32).view(np.int32)))
            ptrs.append(base.data_ptr() + 4 * off)
        out = torch.full((GUARD + oo + n + GUARD,), SENT32 - (1 << 32), dtype=torch.int32, device="cuda")
        n0 = env.ctx.launch_count()
        ix.count_dev(n, ptrs[0], ptrs[1], ptrs[2], m, out.data_ptr() + 4 * (GUARD + oo))
        k = env.ctx.launch_count() - n0
        host = out.cpu().numpy().view(np.uint32)
    assert (host[:GUARD + oo] == SENT32).all(), "count_dev wrote before its output"
    assert (host[GUARD + oo + n:] == SENT32).all(), "count_dev wrote past its output"
    return host[GUARD + oo:GUARD + oo + n], k


def check_dev(env, ix, o, plan, q, m=0, offsets=(0, 0, 0, 0), want=None, what=""):
    from oracle import oracle as orc
    n = len(q[0])
    p = path(plan, n, m, aligned_in=not any(offsets[:3]), aligned_out=not offsets[3])
    got, k = run_count_dev(env, ix, q, m, offsets)
    assert k == LAUNCHES[p], f"{what}: count_dev {offsets} ran {k} launches, the {p} path is {LAUNCHES[p]}"
    if want is None:
        want = o.count(*q, m, threads=orc.max_threads())
    assert_same(got, want, f"{what}: count_dev {offsets} ({p}, min_overlap {m})")


def both_paths(monkeypatch):
    """GTGPU_COUNT_PARTITION forced to 0 and to 1 in turn."""
    for force in ("0", "1"):
        monkeypatch.setenv("GTGPU_COUNT_PARTITION", force)
        yield force


def grouped(chroms):
    """[(starts, ends)] per chromosome -> (offs, s, e)."""
    offs = np.concatenate([[0], np.cumsum([len(a) for a, _ in chroms])]).astype(np.uint64)
    s = np.concatenate([np.asarray(a, np.int64) for a, _ in chroms] + [np.zeros(0, np.int64)])
    e = np.concatenate([np.asarray(b, np.int64) for _, b in chroms] + [np.zeros(0, np.int64)])
    assert (s >= 0).all() and (e <= U32).all()
    return offs, s.astype(np.uint32), e.astype(np.uint32)


def random_index(rng, n_chroms, n, span, width=3000, empty=()):
    """n random proper intervals over n_chroms chromosomes of `span` bp; the chromosomes in `empty` get none."""
    live = np.array([c for c in range(n_chroms) if c not in empty])
    chr_ = np.sort(rng.choice(live, n))
    s = rng.integers(0, span, n)
    e = np.minimum(s + rng.integers(0, width, n), U32)
    offs = np.searchsorted(chr_, np.arange(n_chroms + 1)).astype(np.uint64)
    return offs, s.astype(np.uint32), e.astype(np.uint32)


def random_queries(rng, n_chroms, n, span, degenerate=0.1, unknown=0.03):
    """Queries over [0, span): a fraction `degenerate` empty or reversed, a fraction `unknown` with unknown chromosome ids."""
    qc = rng.integers(0, n_chroms, n).astype(np.int64)
    k = rng.random(n)
    qc[k < unknown / 3] = n_chroms
    qc[(k >= unknown / 3) & (k < 2 * unknown / 3)] = n_chroms + 1
    qc[(k >= 2 * unknown / 3) & (k < unknown)] = U32
    qs = rng.integers(0, span, n)
    qe = qs + rng.integers(1, 4000, n)
    d = rng.random(n)
    qe = np.where(d < degenerate / 2, qs, qe)                                                   # empty
    qe = np.where((d >= degenerate / 2) & (d < degenerate), np.maximum(qs - rng.integers(1, 900, n), 0), qe)  # reversed
    return qc.astype(np.uint32), qs.astype(np.uint32), np.minimum(qe, U32).astype(np.uint32)


# ---- 1. every rank-LUT word form, on both paths ----------------------------------------------------------------------------
def _in_bin(rng, sigma, k):
    """k in-bin offsets: offset 0, the mask, a duplicate, the rest random."""
    mask = (1 << sigma) - 1
    if k == 0:
        return np.zeros(0, np.int64)
    o = rng.integers(0, mask + 1, k)
    o[0] = 0
    if k > 1:
        o[-1] = mask
    if k > 2:
        o[1] = o[rng.integers(2, k)] if rng.random() < 0.5 else 0
    return np.sort(o)


def _shared_bin(rng, sigma, b, k):
    """k intervals inside bin b: starts and ends both planted there, each end at or after its start."""
    mask = (1 << sigma) - 1
    so = _in_bin(rng, sigma, k)
    eo = so + (rng.integers(0, mask + 1, k) * (mask - so)) // max(mask, 1)
    eo[0] = so[0]
    eo[-1] = mask
    return (b << sigma) + so, (b << sigma) + eo


def word_form_chrom(rng, sigma, groups):
    """Starts and ends of one chromosome in bins of 2^sigma: bin 0 and the last bin crowded in both arrays, and `groups` times
    a run of bins holding 0, 1, ..., rank_inline + 1 and many entries (in a random order) in the starts, followed by such a
    run in the ends with its own order and offsets.  Every end of a run lies after every start of its run, so sorted
    starts and sorted ends pair into proper intervals."""
    R = rank_inline(sigma)
    many = R + 6
    pattern = list(range(R + 2)) + [many]
    s0, e0 = _shared_bin(rng, sigma, 0, many)
    S, E = [s0], [e0]
    b = 1
    for _ in range(groups):
        for k in rng.permutation(pattern):
            S.append((b << sigma) + _in_bin(rng, sigma, int(k)))
            b += 1
        for k in rng.permutation(pattern):
            E.append((b << sigma) + _in_bin(rng, sigma, int(k)))
            b += 1
    s1, e1 = _shared_bin(rng, sigma, b, many + 1)
    S.append(s1)
    E.append(e1)
    S, E = np.sort(np.concatenate(S)), np.sort(np.concatenate(E))
    assert len(S) == len(E) and (S <= E).all() and E[-1] <= U32
    perm = rng.permutation(len(S))  # the build sorts them again
    return S[perm], E[perm]


def word_form_layout(sigma, seed, lin=True):
    """Chromosomes [empty, A, B, empty, C, empty] of word_form_chrom; at sigma = 29 the bins run out (eight per 2^32), so one
    chromosome between empty ones: with lin its starts take 3 LUT words and its ends 5 (rank_lin fits), without 5 and 9
    (it does not)."""
    rng = np.random.default_rng(seed)
    empty = (np.zeros(0, np.int64), np.zeros(0, np.int64))
    if sigma < 29:
        chroms = [empty, word_form_chrom(rng, sigma, 2), word_form_chrom(rng, sigma, 2), empty,
                  word_form_chrom(rng, sigma, 1), empty]
        return grouped(chroms)
    many = 7
    if lin:
        cs, ce = [many, 2], [1, many + 1]   # starts in bins 0-1, ends in bins 2-3
    else:
        cs, ce = [many, 0, 1, 2], [2, 1, 0, many]  # starts in bins 0-3, ends in bins 4-7 (up to 2^32 - 1)
    S = np.concatenate([(b << 29) + _in_bin(rng, 29, k) for b, k in enumerate(cs)])
    E = np.concatenate([((b + len(cs)) << 29) + _in_bin(rng, 29, k) for b, k in enumerate(ce)])
    S, E = np.sort(S), np.sort(E)
    assert (S <= E).all()
    return grouped([empty, (S, E), empty])


def probe_queries(rng, offs, s, e, sigma, n_random=3000):
    """Queries on every chromosome that look up every planted value +-1 in both arrays, every bin edge, the last bin and past
    it, start = 2^32 - 1 (start + 1 wraps); empty and reversed queries; and queries on empty and unknown chromosomes."""
    n_chroms = len(offs) - 1
    qc, qs, qe = [], [], []

    def add(c, a, b):
        a, b = np.asarray(a, np.int64), np.asarray(b, np.int64)
        qc.append(np.full(len(a), c, np.int64))
        qs.append(np.clip(a, 0, U32))
        qe.append(np.clip(b, 0, U32))

    for c in range(n_chroms):
        lo, hi = int(offs[c]), int(offs[c + 1])
        cs, ce = s[lo:hi].astype(np.int64), e[lo:hi].astype(np.int64)
        top = int(max(cs.max(initial=0), ce.max(initial=0)))
        nb = (top >> sigma) + 2
        edges = np.arange(nb + 1, dtype=np.int64) << sigma
        edges = np.concatenate([edges - 1, edges, edges + 1, edges + (1 << sigma) - 1, [0, 1, U32 - 1, U32]])
        # end keys search the starts, start + 1 keys the ends
        ke = np.unique(np.clip(np.concatenate([cs - 1, cs, cs + 1, edges]), 0, U32))
        ks = np.unique(np.clip(np.concatenate([ce - 2, ce - 1, ce, edges - 1, edges]), 0, U32))
        # every end key once, with a start below it where there is one
        add(c, np.maximum(ke - 1 - rng.integers(0, 1 << max(sigma, 4), len(ke)), 0), ke)
        # every start key once, with an end above it (start = 2^32 - 1: an empty query)
        add(c, ks, np.minimum(ks + 1 + rng.integers(0, 1 << max(sigma, 4), len(ks)), U32))
        # random pairs of keys: about a half reversed
        add(c, rng.choice(ks, n_random), rng.choice(ke, n_random))
        add(c, ks[:200], ks[:200])  # empty
    qc, qs, qe = np.concatenate(qc), np.concatenate(qs), np.concatenate(qe)
    # the same intervals on unknown ids
    k = rng.choice(len(qc), 600, replace=False)
    unk = np.array([n_chroms, n_chroms + 1, U32], np.int64)
    qc = np.concatenate([qc, unk[np.arange(600) % 3]])
    qs, qe = np.concatenate([qs, qs[k]]), np.concatenate([qe, qe[k]])
    perm = rng.permutation(len(qc))
    return qc[perm].astype(np.uint32), qs[perm].astype(np.uint32), qe[perm].astype(np.uint32)


SIGMAS = [0, 1, 2, 7, 8, 9, 10, 14, 15, 20, 29]


@pytest.mark.parametrize("sigma", SIGMAS)
def test_rank_word_forms(env, monkeypatch, sigma):
    """Bins with 0 .. rank_inline + 1 and many entries, at offsets 0 and the mask and with duplicates, in the starts and
    independently in the ends; crowded bins first and last in a chromosome, with non-empty and empty neighbours; every
    planted value +-1 and every bin edge as a key, on the direct and the bucketed pass and on the scalar kernel."""
    monkeypatch.setenv("GTGPU_RANK_BINS_PER_INTERVAL", HUGE_BINS)
    monkeypatch.setenv("GTGPU_RANK_SHIFT_EXTRA", str(sigma))
    for lin in ((True, False) if sigma == 29 else (True,)):
        offs, s, e = word_form_layout(sigma, seed=1000 + sigma, lin=lin)
        ix, o, plan = build(env, BITS, offs, s, e)
        assert plan.sigma == sigma and plan.has_lin == lin and plan.proper
        # the layout holds every word form of this shift, in each block (at sigma 29 with rank_lin: in the two together):
        # counts 0 .. rank_inline and crowded bins
        want_forms, union = set(range(plan.inline + 1)) | {7}, set()
        for arr in (s, e):
            forms = set()
            for a, b in zip(offs[:-1].astype(np.int64), offs[1:].astype(np.int64)):
                if b > a:
                    forms |= {int(x) if x <= plan.inline else 7 for x in np.bincount(arr[a:b].astype(np.int64) >> sigma)}
            assert forms == want_forms or (sigma == 29 and lin), (forms, want_forms)
            union |= forms
        assert union == want_forms, (union, want_forms)
        rng = np.random.default_rng(sigma)
        q = probe_queries(rng, offs, s, e, sigma)
        assert (q[1] == U32).any() and (q[1] > q[2]).any() and (q[1] == q[2]).any()
        for force in both_paths(monkeypatch):
            want = check_host(env, ix, o, plan, q, what=f"sigma {sigma} lin {lin} partition {force}")
            check_dev(env, ix, o, plan, q, offsets=(0, 1, 0, 0), want=want, what=f"sigma {sigma} lin {lin}")


@pytest.mark.parametrize("kind", [BITS, AILIST], ids=["bits", "ailist"])
def test_rank_word_forms_ailist_and_min_overlap(env, monkeypatch, kind):
    """The same layout at rank_inline 3 under both index kinds, with min_overlap 0 / 1 (identity) and 2 (walk)."""
    monkeypatch.setenv("GTGPU_RANK_BINS_PER_INTERVAL", HUGE_BINS)
    monkeypatch.setenv("GTGPU_RANK_SHIFT_EXTRA", "9")
    offs, s, e = word_form_layout(9, seed=77)
    ix, o, plan = build(env, kind, offs, s, e)
    q = probe_queries(np.random.default_rng(5), offs, s, e, 9)
    for force in both_paths(monkeypatch):
        for m in (0, 1, 2):
            check_host(env, ix, o, plan, q, m, what=f"kind {kind} partition {force}")


# ---- 2. bucket plans and tile shapes ---------------------------------------------------------------------------------------
TILE_SIGMA = 8
TILE_NB = 340  # bins per chromosome: three chromosomes make 3 x 341 = 1023 starts words, so 256 buckets of 4 words are all in use


@pytest.fixture(scope="module")
def tile_index():
    """Three chromosomes of 4 000 intervals whose starts fill exactly TILE_NB bins of 2^8 (rank shift pinned to 8)."""
    rng = np.random.default_rng(2024)
    chroms = []
    for _ in range(3):
        s = rng.integers(0, TILE_NB << TILE_SIGMA, 4000)
        s[0] = ((TILE_NB - 1) << TILE_SIGMA) + 17
        chroms.append((s, s + rng.integers(0, 2000, 4000)))
    return grouped(chroms)


def _tile_queries(rng, plan, words, n):
    """n staged (count-identity) queries whose end keys fall in the given starts-LUT words."""
    w = rng.choice(np.asarray(words, np.int64), n)
    c = np.searchsorted(plan.lut_cs, w, side="right") - 1
    j = w - plan.lut_cs[c]
    e = (j << plan.sigma) + rng.integers(0, 1 << plan.sigma, n)
    e = np.where(j == plan.nb_cs[c], (plan.nb_cs[c] << plan.sigma) + rng.integers(0, 1 << 20, n), e)  # sentinel word
    e = np.maximum(e, 1)
    s = np.maximum(e - rng.integers(1, 3000, n), 0)
    return c.astype(np.uint32), s.astype(np.uint32), e.astype(np.uint32)


def _walk_only(rng, n_chroms, n, unknown_only=False):
    """Queries nothing of which is staged for count / any: unknown ids, empty and reversed queries (unknown_only: nothing is
    staged for bits_count either)."""
    qc = rng.integers(0, n_chroms, n).astype(np.int64)
    qs = rng.integers(1000, 80_000, n)
    k = rng.integers(0, 3 if unknown_only else 6, n)  # 0-2: unknown ids; 3, 5: reversed; 4: empty
    qc = np.where(k == 0, n_chroms, np.where(k == 1, n_chroms + 1, np.where(k == 2, U32, qc)))
    qe = np.where(k % 2 == 0, qs, np.maximum(qs - rng.integers(1, 900, n), 0))
    return qc.astype(np.uint32), qs.astype(np.uint32), qe.astype(np.uint32)


def _cat(*qs):
    return tuple(np.concatenate([q[i] for q in qs]) for i in range(3))


@pytest.mark.parametrize("buckets", [2, 3, 5, 32, 100, 128, 255, 256])
def test_bucket_plans_and_tiles(env, monkeypatch, tile_index, buckets):
    """GTGPU_COUNT_BUCKETS forced; tiles whose queries all share one bucket (a 4 096-long run), tiles with 8k + 1 queries in
    every bucket (the most padding), tiles with nothing staged (whole, and as a partial last tile), and the batch sizes
    around one tile."""
    monkeypatch.setenv("GTGPU_RANK_BINS_PER_INTERVAL", HUGE_BINS)
    monkeypatch.setenv("GTGPU_RANK_SHIFT_EXTRA", str(TILE_SIGMA))
    monkeypatch.setenv("GTGPU_COUNT_BUCKETS", str(buckets))
    monkeypatch.setenv("GTGPU_COUNT_PARTITION", "1")
    ix, o, plan = build(env, BITS, *tile_index)
    assert plan.sigma == TILE_SIGMA and plan.words_s == 3 * (TILE_NB + 1) and plan.has_lin
    nb, shift = bucket_plan(plan, CP_TILE, env.sm)
    used = sorted({min(w >> shift, nb - 1) for w in range(plan.words_s)})
    assert nb == buckets
    if nb in (2, 256):
        assert len(used) == nb  # the 1 023 starts words reach every bucket
    rng = np.random.default_rng(buckets)
    n_chroms = plan.n_chroms
    # one bucket: a 4 096-long run
    b0 = nb // 2
    words = [w for w in range(plan.words_s) if min(w >> shift, nb - 1) == b0]
    one = _tile_queries(rng, plan, words, CP_TILE)
    assert {bucket_of(plan, nb, shift, c, e_) for c, e_ in zip(one[0], one[2])} == {b0}
    # every bucket in use: 8k + 1 queries each, so every run carries 7 entries of padding
    k = np.full(len(used), (CP_TILE - len(used)) // (8 * len(used)))
    k[:((CP_TILE - len(used)) // 8) - int(k.sum())] += 1
    sizes = 8 * k + 1
    spread = _cat(*[_tile_queries(rng, plan, [w for w in range(plan.words_s) if min(w >> shift, nb - 1) == b], int(n_))
                    for b, n_ in zip(used, sizes)])
    perm = rng.permutation(len(spread[0]))
    spread = tuple(a[perm] for a in spread)
    rest = CP_TILE - len(spread[0])
    assert 0 <= rest < 8
    spread = _cat(spread, _walk_only(rng, n_chroms, rest, unknown_only=True))
    got_b = np.bincount([bucket_of(plan, nb, shift, c, e_) for c, e_ in zip(spread[0][:len(perm)], spread[2][:len(perm)])],
                        minlength=nb)
    assert ((got_b[used] % 8) == 1).all() and len(spread[0]) == CP_TILE
    walk = _walk_only(rng, n_chroms, CP_TILE)
    unknown = _walk_only(rng, n_chroms, CP_TILE, unknown_only=True)
    tail = _walk_only(rng, n_chroms, 1234)
    batch = _cat(one, spread, walk, unknown, spread, one, tail)
    check_host(env, ix, o, plan, batch, what=f"{nb} buckets")
    check_host(env, ix, o, plan, _walk_only(rng, n_chroms, 777, unknown_only=True), what="a partial tile, nothing staged")
    check_host(env, ix, o, plan, _walk_only(rng, n_chroms, 777), what="a partial tile, nothing staged for count")
    span = (TILE_NB + 4) << TILE_SIGMA
    for n in (1, 3, 4, 4095, 4096, 4097):
        check_host(env, ix, o, plan, random_queries(rng, n_chroms, n, span), what=f"{nb} buckets, {n} queries")
    check_dev(env, ix, o, plan, batch, what=f"{nb} buckets, count_dev")


def test_automatic_bucket_plans(env, monkeypatch):
    """The automatic bucket count (32, 64, 128 from the LUT size, n and the SM count) and an index so small that
    bucket_shift is 0."""
    monkeypatch.setenv("GTGPU_COUNT_PARTITION", "1")
    monkeypatch.setenv("GTGPU_RANK_BINS_PER_INTERVAL", HUGE_BINS)
    monkeypatch.setenv("GTGPU_RANK_SHIFT_EXTRA", "4")
    rng = np.random.default_rng(11)
    span = 1 << 21
    offs, s, e = random_index(rng, 4, 20_000, span)
    for c in range(4):
        s[int(offs[c])] = span - 5  # every chromosome's LUT runs to the end of the span
    e = np.maximum(e, s)
    ix, o, plan = build(env, BITS, offs, s, e)
    assert plan.sigma == 4 and plan.has_lin
    reached = {}
    for n in (50_000, 100_000, 200_000, 300_000, 400_000, 500_000, 700_000, 1_000_000, 2_000_000):
        reached.setdefault(bucket_plan(plan, n, env.sm)[0], n)
    assert {32, 64, 128} <= set(reached), reached
    for nb in (32, 64, 128):
        q = random_queries(rng, 4, reached[nb], span)
        check_host(env, ix, o, plan, q, what=f"automatic plan of {nb} buckets")

    monkeypatch.setenv("GTGPU_RANK_SHIFT_EXTRA", "16")
    offs, s, e = random_index(rng, 1, 3000, 1 << 20)
    ix, o, plan = build(env, BITS, offs, s, e)
    nb, shift = bucket_plan(plan, 5000, env.sm)
    assert plan.words_s < nb and shift == 0
    check_host(env, ix, o, plan, random_queries(rng, 1, 5000, 1 << 20), what="bucket_shift 0")


# ---- 3. several rounds per block -------------------------------------------------------------------------------------------
def test_many_rounds_per_block(env, monkeypatch):
    """One seeded batch with n % 4 == 3 against a small index: the direct pass strides count_kernel_x4's grid at least twice
    (prefetch and tail), the bucketed pass runs every block of the stage and unstage grids through several tiles (both
    mbarrier phases, both unstage buffers) and count_runs_kernel through many chunks."""
    rng = np.random.default_rng(3)
    offs, s, e = random_index(rng, 6, 30_000, 2_000_000, empty=(2,))
    ix, o, plan = build(env, BITS, offs, s, e)
    x4_step = 4 * 256 * X4_STRIDE_BLOCKS * env.sm
    resident = 2 * env.sm * CP_TILE  # two 1 024-thread blocks per SM, one tile each per round
    n = max(int(x4_step * 1.03), 3 * resident + 5 * CP_TILE)
    n += (3 - n % 4) % 4
    assert n % 4 == 3 and n > x4_step and n > 3 * resident
    q = random_queries(rng, 6, n, 2_000_000)
    for force in both_paths(monkeypatch):
        assert path(plan, n) == ("bucketed" if force == "1" else "x4")
        check_host(env, ix, o, plan, q, what=f"{n} queries, partition {force}")


# ---- 4. alignment, the scalar kernel and stray writes ----------------------------------------------------------------------
OFFSETS = [(0, 0, 0, 0)] + [tuple(k if i == j else 0 for i in range(4)) for j in range(4) for k in (1, 2, 3)] + \
          [(k, k, k, k) for k in (1, 2, 3)]


@pytest.fixture(scope="module")
def word_form_9():
    return word_form_layout(9, seed=909)


def test_alignment_and_scalar_kernel(env, monkeypatch, word_form_9):
    """gtgpu_count_dev with each of chr, start, end, out offset by 1, 2 and 3 elements, one at a time and all together:
    unaligned input runs count_kernel even when partitioning is forced; an unaligned output alone runs the bucketed pass with
    element stores when it is forced and count_kernel when it is not.  Sentinel guard bands catch any stray write."""
    from oracle import oracle as orc
    monkeypatch.setenv("GTGPU_RANK_BINS_PER_INTERVAL", HUGE_BINS)
    monkeypatch.setenv("GTGPU_RANK_SHIFT_EXTRA", "9")
    offs, s, e = word_form_9
    ix, o, plan = build(env, BITS, offs, s, e)
    rng = np.random.default_rng(4)
    probes = probe_queries(rng, offs, s, e, 9)
    th = orc.max_threads()
    for n in (0, 1, 2, 3, 5, 4097, len(probes[0])):
        q = tuple(a[:n] for a in probes)
        want = o.count(*q, 0, threads=th)
        for force in both_paths(monkeypatch):
            for off in OFFSETS:
                check_dev(env, ix, o, plan, q, offsets=off, want=want, what=f"n {n}, partition {force}")
    # a batch across the scalar kernel's grid-stride loop (and several tiles of the bucketed pass)
    n = 256 * X4_STRIDE_BLOCKS * env.sm * 2 + 3
    reps = -(-n // len(probes[0]))
    q = tuple(np.tile(a, reps)[:n] for a in probes)
    want = o.count(*q, 0, threads=th)
    for force in both_paths(monkeypatch):
        for off in ((1, 0, 0, 0), (0, 0, 0, 3), (2, 2, 2, 2)):
            check_dev(env, ix, o, plan, q, offsets=off, want=want, what=f"{n} queries, partition {force}")


# ---- 5. more than 256 chromosomes ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n_chroms", [300, 2000])
def test_many_chromosomes(env, monkeypatch, n_chroms):
    """The stage kernel keeps rank_lin of the first 256 chromosomes in shared memory and reads the rest from global memory:
    query ids below 256, at 255 and 256, above, and unknown ids n_chroms, n_chroms + 1 and 2^32 - 1, on both paths."""
    rng = np.random.default_rng(n_chroms)
    span = 1 << 20
    empty = set(rng.choice(n_chroms, n_chroms // 20, replace=False).tolist()) - {255, 256}
    offs, s, e = random_index(rng, n_chroms, 30 * n_chroms, span, width=20_000, empty=empty)
    ix, o, plan = build(env, BITS, offs, s, e)
    assert plan.has_lin
    q = random_queries(rng, n_chroms, 150_000, span)
    qc = q[0].astype(np.int64)
    pick = rng.random(len(qc))
    qc = np.where(pick < 0.1, 255, np.where(pick < 0.2, 256, np.where(pick < 0.25, n_chroms - 1, qc)))
    qc[:3] = [n_chroms, n_chroms + 1, U32]
    q = (qc.astype(np.uint32), q[1], q[2])
    assert (q[0] < 256).any() and (q[0] > 256).sum() > 1000
    for force in both_paths(monkeypatch):
        check_host(env, ix, o, plan, q, what=f"{n_chroms} chromosomes, partition {force}")


# ---- 6. the walk and the launcher's refusals -------------------------------------------------------------------------------
def _nested_index(rng, n_chroms, n, span):
    """Intervals with some long ones over many short ones: an AIList of several components."""
    chr_ = np.sort(rng.integers(0, n_chroms, n))
    s = rng.integers(0, span, n)
    w = np.where(rng.random(n) < 0.1, rng.integers(5000, 80_000, n), rng.integers(1, 400, n))
    offs = np.searchsorted(chr_, np.arange(n_chroms + 1)).astype(np.uint64)
    return offs, s.astype(np.uint32), np.minimum(s + w, U32).astype(np.uint32)


@pytest.mark.parametrize("kind", [BITS, AILIST], ids=["bits", "ailist"])
def test_min_overlap_and_components(env, monkeypatch, kind):
    """min_overlap 0, 1, 2 and 50: above 1 a call is always direct and walks; AIList indexes with several components."""
    rng = np.random.default_rng(60 + kind)
    offs, s, e = _nested_index(rng, 5, 20_000, 300_000)
    ix, o, plan = build(env, kind, offs, s, e)
    if kind == AILIST:
        assert ix.info()["max_components"] >= 2
    q = random_queries(rng, 5, 20_000, 300_000, degenerate=0.2)
    for force in both_paths(monkeypatch):
        for m in (0, 1, 2, 50):
            check_host(env, ix, o, plan, q, m, what=f"partition {force}")
            if m == 50:
                assert path(plan, len(q[0]), m) == "x4"


def test_improper_index(env, monkeypatch):
    """An index with some start > end: direct and walked for count / any (the identity would be wrong), direct with the
    identity for bits_count, even when partitioning is forced."""
    rng = np.random.default_rng(61)
    offs, s, e = random_index(rng, 4, 10_000, 200_000)
    flip = rng.random(len(s)) < 0.05
    e = np.where(flip, np.maximum(s.astype(np.int64) - rng.integers(1, 500, len(s)), 0), e).astype(np.uint32)
    ix, o, plan = build(env, BITS, offs, s, e)
    assert not plan.proper and not ix.info()["proper"]
    q = random_queries(rng, 4, 30_000, 200_000)
    for force in both_paths(monkeypatch):
        assert path(plan, len(q[0])) == "x4"
        for m in (0, 2):
            check_host(env, ix, o, plan, q, m, what=f"improper, partition {force}")
        check_dev(env, ix, o, plan, q, offsets=(1, 1, 1, 1), what="improper")


@pytest.mark.parametrize("lut_shift", ["0", None, "31"])
@pytest.mark.parametrize("kind", [BITS, AILIST], ids=["bits", "ailist"])
def test_segment_lut_shift(env, monkeypatch, kind, lut_shift):
    """GTGPU_LUT_SHIFT 0, default and 31 for the walk's segment LUTs (lut_lower_bound, including its past-the-last-bin
    return): empty and reversed queries, min_overlap 2 and keys beyond every interval."""
    if lut_shift is not None:
        monkeypatch.setenv("GTGPU_LUT_SHIFT", lut_shift)
    rng = np.random.default_rng(62 + kind)
    offs, s, e = _nested_index(rng, 3, 8000, 150_000)
    ix, o, plan = build(env, kind, offs, s, e)
    if lut_shift is not None:
        assert ix.info()["lut_shift"] == int(lut_shift)
    q = random_queries(rng, 3, 20_000, 400_000, degenerate=0.3)
    qe = q[2].copy()
    qe[:100] = U32
    q = (q[0], q[1], qe)
    for force in both_paths(monkeypatch):
        for m in (0, 2):
            check_host(env, ix, o, plan, q, m, what=f"lut shift {lut_shift}, partition {force}")


@pytest.mark.parametrize("kind", [BITS, AILIST], ids=["bits", "ailist"])
def test_empty_indexes(env, monkeypatch, kind):
    """An index without chromosomes (no rank LUT: direct) and one whose chromosomes are all empty (sentinel words only)."""
    rng = np.random.default_rng(63)
    for offs in (np.zeros(1, np.uint64), np.zeros(4, np.uint64)):
        ix, o, plan = build(env, kind, offs, np.zeros(0, np.uint32), np.zeros(0, np.uint32))
        assert plan.has_lin and plan.lut_len == 2 * plan.n_chroms
        q = random_queries(rng, max(plan.n_chroms, 1), 5000, 100_000, degenerate=0.2)
        for force in both_paths(monkeypatch):
            want = check_host(env, ix, o, plan, q, what=f"{plan.n_chroms} empty chromosomes, partition {force}")
            assert not want.any()
            check_dev(env, ix, o, plan, q, offsets=(0, 0, 0, 1), want=want, what="empty index")


def test_bits_count_refuses_ailist(env):
    from gtars_b200 import ffi
    offs, s, e = random_index(np.random.default_rng(64), 2, 100, 10_000)
    ix, _, _ = build(env, AILIST, offs, s, e)
    with pytest.raises(ffi.GtarsGpuError):
        ix.bits_count(np.zeros(4, np.uint32), np.zeros(4, np.uint32), np.ones(4, np.uint32))


def test_automatic_selection(env, monkeypatch):
    """Without GTGPU_COUNT_PARTITION the bucketed pass runs for a rank LUT beyond 64 MiB and at least 4 Mi queries: 3 launches
    at n = 4 Mi, 1 at 4 Mi - 4, and 1 for the same database with a LUT under 64 MiB."""
    monkeypatch.delenv("GTGPU_COUNT_PARTITION", raising=False)
    rng = np.random.default_rng(65)
    span = 1 << 25
    offs, s, e = random_index(rng, 2, 1 << 20, span)
    qs = {n: random_queries(rng, 2, n, span) for n in (4 << 20, (4 << 20) - 4)}
    for bins, big in (("16", True), (None, False)):
        if bins is None:
            monkeypatch.delenv("GTGPU_RANK_BINS_PER_INTERVAL", raising=False)
        else:
            monkeypatch.setenv("GTGPU_RANK_BINS_PER_INTERVAL", bins)
        ix, o, plan = build(env, BITS, offs, s, e)
        assert (plan.lut_len * 8 > 64 << 20) == big and plan.has_lin
        for n, q in qs.items():
            assert path(plan, n) == ("bucketed" if big and n >= 4 << 20 else "x4")
            check_host(env, ix, o, plan, q, what=f"rank LUT {plan.lut_len * 8 >> 20} MiB, {n} queries")
        del ix


# ---- 7. the 2^31 guard -----------------------------------------------------------------------------------------------------
def test_two_pow_31_guard(env, monkeypatch):
    """n = 2^31 is refused by the bucketed pass (its staged positions are 32-bit) and runs direct, exactly, even when
    partitioning is forced; n = 2^31 - 4 with 256 buckets reaches the largest staged offsets (tile x cap near 3.2e9).  The
    queries repeat one period, generated on the device; the expected counts are the period's, tiled."""
    import torch
    free, _ = torch.cuda.mem_get_info()
    if free < 100e9:
        pytest.skip(f"needs about 80 GB of device memory, {free / 1e9:.0f} GB free")
    rng = np.random.default_rng(66)
    offs, s, e = random_index(rng, 3, 20_000, 1_000_000)
    ix, o, plan = build(env, BITS, offs, s, e)
    P = 4093
    pq = random_queries(rng, 3, P, 1_000_000, degenerate=0.1)
    p_want = o.count(*pq, 0)
    assert p_want.any()
    monkeypatch.setenv("GTGPU_COUNT_PARTITION", "1")
    monkeypatch.setenv("GTGPU_COUNT_BUCKETS", "256")
    N = 1 << 31
    with torch.cuda.stream(env.stream):
        def periodic(a, n):
            t = torch.empty(n, dtype=torch.int32, device="cuda")
            rows = n // P
            src = torch.from_numpy(np.ascontiguousarray(a, np.uint32).view(np.int32)).to("cuda")
            t[:rows * P].view(rows, P).copy_(src.expand(rows, P))
            t[rows * P:].copy_(src[:n - rows * P])
            return t
        d_q = [periodic(a, N) for a in pq]
        want = periodic(p_want, N)
        out = torch.empty(N, dtype=torch.int32, device="cuda")
        for n in (N, N - 4):
            p = path(plan, n)
            assert p == ("x4" if n == N else "bucketed")
            out.fill_(SENT32 - (1 << 32))
            n0 = env.ctx.launch_count()
            ix.count_dev(n, d_q[0].data_ptr(), d_q[1].data_ptr(), d_q[2].data_ptr(), 0, out.data_ptr())
            assert env.ctx.launch_count() - n0 == LAUNCHES[p]
            bad = int((out[:n] != want[:n]).sum().item())
            assert bad == 0, f"{n} queries ({p}): {bad} counts differ"
            if n < N:
                assert (out[n:] == SENT32 - (1 << 32)).all().item(), "written past the output"
    env.stream.synchronize()
    del d_q, want, out
    torch.cuda.empty_cache()
