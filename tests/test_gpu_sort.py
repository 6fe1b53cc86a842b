"""The device sort and scan primitives of sort.cu against exact numpy references, and their callers against the oracle.

Part 1 calls radix_sort_pairs, radix_group_values, exclusive_scan<u32 / u64> and inclusive_max_scan_u64 directly, through
tests/sort_shim.cpp (they are not in the C ABI): every digit plan radix_plan can choose, the three scatter tile shapes
(GTGPU_RS_SHAPE) at tile edges, the 4-byte cp.async staging of misaligned full tiles, the looping scan spine, element counts
known only on the device, and the packed group-by at every upper-digit width and at the packing boundary.  Output buffers
start out filled with sentinels and carry a guard band, so a missing write or a write past the end shows.

Part 2 runs the callers through the C ABI against the CPU oracle at the plans they choose: fragment tokenization (host and
device-resident, every pair-sort plan under every tile shape, the group-by / pair-sort switch set by the token width),
barcode scoring at peak-id widths on plan edges, and the stable (name, start) sort of gtgpu_parse_bed over the whole u32 range.
"""
import ctypes as C
import os
import subprocess
import types
import zlib

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
SHAPE_TILE = {0: 8192, 1: 6144, 2: 16384}  # scatter tile of each GTGPU_RS_SHAPE (threads x rounds, sort.cu RS_SHAPES)
SCAN_TILE = 2048                            # elements per scan tile; the spine scans 256 tile sums per round
GUARD = 64
SENT32 = 0xA5A5A5A5
SENT64 = 0xA5A5A5A5A5A5A5A5
# radix_plan: bits -> (passes, digit width)
PLANS = {1: (1, 8), 8: (1, 8), 9: (1, 9), 10: (2, 8), 16: (2, 8), 17: (2, 9), 18: (2, 9), 19: (3, 8), 24: (3, 8), 25: (3, 9),
         27: (3, 9), 28: (4, 8), 32: (4, 8)}


def _bits_for(n_values):
    b = 1
    while (1 << b) < n_values:
        b += 1
    return b


# ---- harness ---------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def env():
    """One context on a torch stream; every primitive runs on it (they never select a device themselves: device 0)."""
    import torch
    from gtars_b200 import ffi
    stream = torch.cuda.Stream()
    ctx = ffi.Context(0, stream=stream.cuda_stream)
    yield types.SimpleNamespace(ctx=ctx, stream=stream)
    stream.synchronize()
    ctx.close()


@pytest.fixture(scope="module")
def shim(tmp_path_factory):
    """tests/sort_shim.cpp built with g++ against the package's libgtars_gpu.so and loaded with ctypes."""
    from gtars_b200 import ffi
    ffi.lib()
    libdir = os.path.dirname(os.path.abspath(ffi.LIB_PATH))
    out = str(tmp_path_factory.mktemp("sort_shim") / "libsort_shim.so")
    env = dict(os.environ)
    env.pop("CXX", None)
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-o", out, os.path.join(HERE, "sort_shim.cpp"),
                           "-L" + libdir, "-lgtars_gpu", "-Wl,-rpath," + libdir], env=env)
    L = C.CDLL(out)
    vp, u64, i32, u32, sz = C.c_void_p, C.c_uint64, C.c_int32, C.c_uint32, C.c_size_t
    sigs = {
        "shim_exclusive_scan_temp_bytes": (sz, [u64, sz]),
        "shim_exclusive_scan_u32": (i32, [vp, vp, vp, u64, vp]),
        "shim_exclusive_scan_u64": (i32, [vp, vp, vp, u64, vp]),
        "shim_inclusive_max_scan_u64": (i32, [vp, vp, vp, u64, vp]),
        "shim_radix_sort_temp_bytes": (sz, [u64]),
        "shim_radix_sort_pairs": (i32, [vp, u64, vp, vp, vp, vp, C.c_int, vp, vp, vp]),
        "shim_radix_plan": (None, [C.c_int, vp, vp]),
        "shim_radix_group_fits": (i32, [u32, u32]),
        "shim_radix_group_temp_bytes": (sz, [u64, u32]),
        "shim_radix_group_values": (i32, [vp, u64, vp, vp, vp, vp, u32, u32, vp, vp, vp, vp]),
    }
    for name, (res, args) in sigs.items():
        fn = getattr(L, name)
        fn.restype, fn.argtypes = res, args
    return L


def _ok(status):
    from gtars_b200 import ffi
    assert status == 0, ffi.lib().gtgpu_last_error().decode(errors="replace")


def _buf(a, lead=0, wide=False):
    """Device copy of `a` behind `lead` sentinel elements and ahead of GUARD more."""
    import torch
    a = np.ascontiguousarray(a, np.uint64 if wide else np.uint32)
    t = torch.full((lead + len(a) + GUARD,), (SENT64 if wide else SENT32) - (1 << (64 if wide else 32)),
                   dtype=torch.int64 if wide else torch.int32, device="cuda")
    if len(a):
        t[lead:lead + len(a)] = torch.from_numpy(a.view(np.int64 if wide else np.int32)).to("cuda")
    return t


def _empty(n, lead=0, wide=False):
    return _buf(np.full(n, SENT64 if wide else SENT32, np.uint64 if wide else np.uint32), lead, wide)


def _ptr(t, lead=0):
    return t.data_ptr() + lead * t.element_size()


def _host(t):
    return t.cpu().numpy().view(np.uint64 if t.element_size() == 8 else np.uint32)


def _temp(nbytes):
    import torch
    return torch.empty(max(int(nbytes), 16), dtype=torch.uint8, device="cuda")


def _run(env, fn, *args):
    """Call a primitive on the ctx stream after everything torch queued, and wait for it."""
    import torch
    torch.cuda.synchronize()
    _ok(fn(*args))
    env.stream.synchronize()


# ---- radix_sort_pairs ------------------------------------------------------------------------------------------------------
def _sort(env, shim, keys, bits, lead=0, dn=None):
    """radix_sort_pairs of (keys, iota) over n = len(keys) (the capacity when dn is given), checked against a stable numpy
    argsort of the first dn (or n) keys' low `bits` bits: keys keep all their bits, values are the permutation, both buffer
    pairs hold exactly what they held before outside [lead, lead + count), and the result lies in the buffer the pass
    count's parity names."""
    import torch
    keys = np.ascontiguousarray(keys, np.uint32)
    n = len(keys)
    count = n if dn is None else dn
    ka, va = _buf(keys, lead), _buf(np.arange(n, dtype=np.uint32), lead)
    kb, vb = _empty(n, lead), _empty(n, lead)
    before = [_host(t) for t in (ka, va, kb, vb)]
    tmp = _temp(shim.shim_radix_sort_temp_bytes(n))
    d_n = torch.tensor([dn], dtype=torch.int64, device="cuda") if dn is not None else None
    in_b = C.c_int(-1)
    _run(env, shim.shim_radix_sort_pairs, env.ctx._h, n, _ptr(ka, lead), _ptr(va, lead), _ptr(kb, lead), _ptr(vb, lead), bits,
         tmp.data_ptr(), C.byref(in_b), d_n.data_ptr() if d_n is not None else None)
    assert in_b.value == PLANS[bits][0] % 2
    after = [_host(t) for t in (ka, va, kb, vb)]
    for a, b in zip(before, after):  # nothing outside the counted elements moved, in either buffer pair
        assert np.array_equal(a[:lead], b[:lead])
        assert np.array_equal(a[lead + count:], b[lead + count:])
    mask = np.uint32(0xFFFFFFFF if bits >= 32 else (1 << bits) - 1)
    order = np.argsort(keys[:count] & mask, kind="stable")
    rk, rv = (after[2], after[3]) if in_b.value else (after[0], after[1])
    assert np.array_equal(rv[lead:lead + count], order.astype(np.uint32))
    assert np.array_equal(rk[lead:lead + count], keys[:count][order])


def _keys(dist, n, bits, rng):
    mask = (1 << bits) - 1
    u = rng.integers(0, 1 << bits, n, dtype=np.uint64)
    if dist == "uniform":
        k = u
    elif dist == "equal":
        k = np.full(n, rng.integers(0, 1 << bits) & mask, np.uint64)
    elif dist == "alternating":
        a, b = rng.integers(0, 1 << bits, 2)
        k = np.where(np.arange(n) % 2 == 0, a, b).astype(np.uint64)
    elif dist == "sorted":
        k = np.sort(u)
    elif dist == "reversed":
        k = np.sort(u)[::-1]
    elif dist == "top_digit":  # the low digits of every key are one constant: every pass but the last sorts pure ties
        passes, width = PLANS[bits]
        shift = (passes - 1) * width
        low = int(rng.integers(0, 1 << shift)) if shift else 0
        k = (rng.integers(0, 1 << (bits - shift), n, dtype=np.uint64) << np.uint64(shift)) | np.uint64(low)
    elif dist == "high_bits":  # bits above `bits` set at random: the sort ignores them and keeps them (below 8 bits, the
        # one 8-bit digit reads bits [0, 8): only bits from 8 up are ignored there)
        k = u | (rng.integers(0, 1 << 32, n, dtype=np.uint64) & np.uint64(~((1 << max(bits, 8)) - 1) & 0xFFFFFFFF))
    else:
        raise ValueError(dist)
    return k.astype(np.uint32)


def test_radix_plan_table(shim):
    """The digit plans radix_plan chooses: as few passes as 9-bit digits allow, 8-bit digits where they suffice."""
    for bits, plan in PLANS.items():
        p, w = C.c_int(), C.c_int()
        shim.shim_radix_plan(bits, C.byref(p), C.byref(w))
        assert (p.value, w.value) == plan, bits


DISTS = ["uniform", "equal", "alternating", "sorted", "reversed", "top_digit", "high_bits"]


@pytest.mark.parametrize("dist", DISTS)
@pytest.mark.parametrize("bits", sorted(PLANS))
def test_radix_sort_every_plan(env, shim, bits, dist):
    """Every digit plan at its edges, every key distribution, over three full tiles and a partial one (default shape)."""
    rng = np.random.default_rng(zlib.crc32(f"plan/{bits}/{dist}".encode()))
    _sort(env, shim, _keys(dist, 3 * 8192 + 17, bits, rng), bits)


@pytest.mark.parametrize("shape", [0, 1, 2])
@pytest.mark.parametrize("where", ["1", "31", "33", "T-1", "T", "T+1", "3T", "3T+17"])
def test_radix_sort_tile_shapes(env, shim, monkeypatch, shape, where):
    """Each scatter tile shape at the element counts around its tile: a lone element, partial warps, a partial tile, exactly
    full tiles (the FULL instantiation) and a partial last tile; keys with many ties across warps (stability between warps)
    and all-equal keys (one digit fills the tile: the per-warp counters reach their largest values)."""
    T = SHAPE_TILE[shape]
    n = {"1": 1, "31": 31, "33": 33, "T-1": T - 1, "T": T, "T+1": T + 1, "3T": 3 * T, "3T+17": 3 * T + 17}[where]
    monkeypatch.setenv("GTGPU_RS_SHAPE", str(shape))
    rng = np.random.default_rng(zlib.crc32(f"shape/{shape}/{where}".encode()))
    _sort(env, shim, (rng.integers(0, 97, n) * 1351).astype(np.uint32), 17)   # 2 x 9: ties in both digits
    _sort(env, shim, (rng.integers(0, 5, n) * 0x01010101).astype(np.uint32), 32)   # 4 x 8
    _sort(env, shim, _keys("equal", n, 9, rng), 9)


@pytest.mark.parametrize("bits", [18, 27])
def test_radix_sort_past_one_spine_round(env, shim, bits):
    """More than 1 024 tiles of 9-bit digits: the bucket table has more than 256 x 2 048 entries, so the scan spine loops."""
    n = 8_388_608 + 8_193
    assert (n + 8191) // 8192 * 512 > 256 * SCAN_TILE
    rng = np.random.default_rng(bits)
    keys = rng.integers(0, 1 << bits, n, dtype=np.uint64).astype(np.uint32)
    keys[rng.random(n) < 0.25] = 12345  # a heavy digit
    _sort(env, shim, keys, bits)


@pytest.mark.parametrize("shape", [0, 1, 2])
@pytest.mark.parametrize("bits", [9, 17, 27])
def test_radix_sort_misaligned_buffers(env, shim, monkeypatch, shape, bits):
    """Key and value pointers one element past 16-byte alignment: full tiles are staged with 4-byte cp.async copies."""
    monkeypatch.setenv("GTGPU_RS_SHAPE", str(shape))
    rng = np.random.default_rng(zlib.crc32(f"mis/{shape}/{bits}".encode()))
    n = 3 * SHAPE_TILE[shape] + 17
    _sort(env, shim, (rng.integers(0, 1 << bits, n) // 7 * 7).astype(np.uint32), bits, lead=1)


@pytest.mark.parametrize("shape", [0, 2])
@pytest.mark.parametrize("bits", [9, 17, 27])
@pytest.mark.parametrize("which", ["0", "1", "T", "cap-1"])
def test_radix_sort_device_count(env, shim, monkeypatch, shape, bits, which):
    """The element count only the device knows (*d_n <= n): the first *d_n keys are sorted, nothing past them is written."""
    monkeypatch.setenv("GTGPU_RS_SHAPE", str(shape))
    T = SHAPE_TILE[shape]
    n = 3 * T + 100
    dn = {"0": 0, "1": 1, "T": T, "cap-1": n - 1}[which]
    rng = np.random.default_rng(zlib.crc32(f"dn/{shape}/{bits}/{which}".encode()))
    _sort(env, shim, rng.integers(0, 1 << bits, n, dtype=np.uint64).astype(np.uint32), bits, dn=dn)


# ---- radix_group_values ----------------------------------------------------------------------------------------------------
def _group_split(n_keys):
    """(upper digit bits hw, low digit width w) of the packed group-by for n_keys keys: two passes of 8 bits for 10-16 key
    bits, of 9 bits for 17 and 18."""
    bits = _bits_for(n_keys)
    assert 10 <= bits <= 18
    w = 9 if bits > 16 else 8
    return bits - w, w


def _group(env, shim, keys, vals, n_keys, max_val, dn=None):
    """radix_group_values over n_cap = len(keys), checked against a stable argsort by key and a cumulative bincount."""
    import torch
    keys, vals = np.ascontiguousarray(keys, np.uint32), np.ascontiguousarray(vals, np.uint32)
    n_cap = len(keys)
    assert shim.shim_radix_group_fits(n_keys, max_val)
    d_k, d_v = _buf(keys), _buf(vals)
    packed, out = _empty(n_cap), _empty(n_cap)
    offs, total = _empty(n_keys + 1, wide=True), _empty(1, wide=True)
    tmp = _temp(shim.shim_radix_group_temp_bytes(n_cap, n_keys))
    d_n = torch.tensor([dn], dtype=torch.int64, device="cuda") if dn is not None else None
    _run(env, shim.shim_radix_group_values, env.ctx._h, n_cap, _ptr(d_k), _ptr(d_v), _ptr(packed), _ptr(out), n_keys, max_val,
         tmp.data_ptr(), d_n.data_ptr() if d_n is not None else None, _ptr(offs), _ptr(total))
    count = n_cap if dn is None else min(dn, n_cap)
    h_tot, h_out, h_off = _host(total), _host(out), _host(offs)
    assert int(h_tot[0]) == (0xFFFFFFFFFFFFFFFF if dn is not None and dn > n_cap else count)
    assert (h_tot[1:] == SENT64).all() and (h_off[n_keys + 1:] == SENT64).all()
    assert (h_out[count:] == SENT32).all()
    assert np.array_equal(_host(d_k)[:n_cap], keys) and np.array_equal(_host(d_v)[:n_cap], vals)  # inputs only read
    order = np.argsort(keys[:count], kind="stable")
    assert np.array_equal(h_out[:count], vals[:count][order])
    ref = np.zeros(n_keys + 1, np.uint64)
    ref[1:] = np.cumsum(np.bincount(keys[:count], minlength=n_keys))
    assert np.array_equal(h_off[:n_keys + 1], ref)


GROUP_KEYS = [513, 1024, 1025, 4097, 65_536, 65_537, 131_072, 131_073, 262_144]
GROUP_PATTERNS = ["uniform", "skewed", "missing", "single", "small", "iota_vals"]


@pytest.mark.parametrize("pattern", GROUP_PATTERNS)
@pytest.mark.parametrize("n_keys", GROUP_KEYS)
def test_group_values(env, shim, n_keys, pattern):
    """The packed group-by at upper-digit widths hw = 2, 3, 5, 8, 9 (low digits of 8 and 9 bits).  Values reach max_val,
    chosen so the packed word is exactly 32 bits wide (bit 31 in use) — one more value bit must leave the group-by."""
    hw, w = _group_split(n_keys)
    rng = np.random.default_rng(zlib.crc32(f"group/{n_keys}/{pattern}".encode()))
    n = 5000 if pattern == "small" else max(3 * n_keys, 200_003)
    keys = rng.integers(0, n_keys, n).astype(np.uint32)
    if pattern == "skewed":  # half the elements share low digit 0: many pass-2 tiles lie inside it, the rest cross boundaries
        hi = rng.integers(0, (n_keys - 1 >> w) + 1, n).astype(np.uint32) << np.uint32(w)
        keys = np.where(rng.random(n) < 0.5, hi, (rng.integers(0, n_keys, n) ** 2 // n_keys)).astype(np.uint32)
    elif pattern == "missing":  # about a tenth of the keys, the last one among them, never occur
        absent = rng.random(n_keys) < 0.1
        absent[-1] = True
        keys = rng.choice(np.flatnonzero(~absent), n).astype(np.uint32)
    elif pattern == "single":
        keys = np.full(n, n_keys // 3, np.uint32)
    if pattern == "iota_vals":
        max_val = n - 1
        vals = np.arange(n, dtype=np.uint32)
    else:
        max_val = (1 << (32 - hw)) - 1
        assert not shim.shim_radix_group_fits(n_keys, max_val + 1)
        vals = rng.integers(0, max_val + 1, n, dtype=np.uint64).astype(np.uint32)
        vals[rng.random(n) < 0.05] = max_val
    _group(env, shim, keys, vals, n_keys, max_val)


@pytest.mark.parametrize("n_keys", [4097, 131_073])
@pytest.mark.parametrize("which", ["0", "1", "cap-1000", "over"])
def test_group_values_device_count(env, shim, n_keys, which):
    """*d_n below the capacity groups the first *d_n elements and writes nothing past them; *d_n above it reports ~0."""
    rng = np.random.default_rng(zlib.crc32(f"groupdn/{n_keys}/{which}".encode()))
    n = 100_000
    dn = {"0": 0, "1": 1, "cap-1000": n - 1000, "over": n + 5}[which]
    keys = rng.integers(0, n_keys, n).astype(np.uint32)
    vals = rng.integers(0, 1 << 20, n).astype(np.uint32)
    _group(env, shim, keys, vals, n_keys, (1 << 20) - 1, dn=dn)


# ---- scans -----------------------------------------------------------------------------------------------------------------
SCAN_NS = [1, 2047, 2048, 2049, 256 * 2048, 256 * 2048 + 1, 3_000_017]


@pytest.mark.parametrize("n", SCAN_NS)
def test_exclusive_scan(env, shim, n):
    """exclusive_scan<u32> wrapping modulo 2^32 and exclusive_scan<u64> with sums far past 2^32, against numpy cumsums."""
    rng = np.random.default_rng(n)
    for wide, fn in ((False, shim.shim_exclusive_scan_u32), (True, shim.shim_exclusive_scan_u64)):
        dt = np.uint64 if wide else np.uint32
        a = rng.integers(0, 1 << (40 if wide else 32), n, dtype=np.uint64).astype(dt)
        d_in, d_out = _buf(a, wide=wide), _empty(n, wide=wide)
        tmp = _temp(shim.shim_exclusive_scan_temp_bytes(n, 8 if wide else 4))
        _run(env, fn, env.ctx._h, _ptr(d_in), _ptr(d_out), n, tmp.data_ptr())
        ref = np.zeros(n, dt)
        ref[1:] = np.cumsum(a[:-1], dtype=dt)
        got = _host(d_out)
        assert np.array_equal(got[:n], ref)
        assert (got[n:] == (SENT64 if wide else SENT32)).all()
        if wide and n > 4096:
            assert int(ref[-1]) > 1 << 32
        elif not wide and n > 4096:
            assert int(np.sum(a, dtype=np.uint64)) > 1 << 32  # the u32 scan wrapped


@pytest.mark.parametrize("in_place", [False, True], ids=["out_of_place", "in_place"])
@pytest.mark.parametrize("n", SCAN_NS)
def test_inclusive_max_scan(env, shim, n, in_place):
    """inclusive_max_scan_u64 over (segment << 32 | value) words as the index and IGD builders use it (igd.cu: in place)."""
    rng = np.random.default_rng(n + in_place)
    seg = np.cumsum(rng.random(n) < 0.001).astype(np.uint64)
    a = (seg << np.uint64(32)) | rng.integers(0, 1 << 32, n, dtype=np.uint64)
    d_in = _buf(a, wide=True)
    d_out = d_in if in_place else _empty(n, wide=True)
    tmp = _temp(shim.shim_exclusive_scan_temp_bytes(n, 8))
    _run(env, shim.shim_inclusive_max_scan_u64, env.ctx._h, _ptr(d_in), _ptr(d_out), n, tmp.data_ptr())
    got = _host(d_out)
    assert np.array_equal(got[:n], np.maximum.accumulate(a))
    assert (got[n:] == SENT64).all()


# ---- part 2: the callers through the C ABI ---------------------------------------------------------------------------------
N_CHROMS = 3


def _universe(env, rng, n, max_val):
    """A Bits index of n random intervals whose vals reach max_val, and the oracle index of the same intervals."""
    from gtars_b200 import ffi
    from oracle import oracle as orc
    chr_ = np.sort(rng.integers(0, N_CHROMS, n))
    s = rng.integers(0, 2_000_000, n).astype(np.uint32)
    e = (s + rng.integers(1, 3000, n)).astype(np.uint32)
    v = rng.integers(0, max_val + 1, n, dtype=np.uint64).astype(np.uint32)
    v[rng.integers(0, n, 8)] = max_val
    offs = np.searchsorted(chr_, np.arange(N_CHROMS + 1)).astype(np.uint64)
    return ffi.Index(env.ctx, ffi.KIND_BITS, offs, s, e, v), orc.Index(ffi.KIND_BITS, offs, s, e, v)


def _fragments(rng, n, n_bc):
    qc = rng.integers(0, N_CHROMS + 1, n).astype(np.uint32)  # id N_CHROMS is unknown: an unk token
    qs = rng.integers(0, 2_010_000, n).astype(np.uint32)
    qe = (qs + rng.integers(1, 1500, n)).astype(np.uint32)
    bc = rng.integers(0, n_bc, n).astype(np.uint32)
    bc[rng.integers(0, n, 3)] = n_bc - 1  # the last barcode occurs
    return qc, qs, qe, bc


# name: (n_barcodes, fragments, largest index val, unk_id, packed group-by?)
FRAG_CASES = {
    "bc1": (1, 40_000, 1 << 20, 5000, False),                        # 1 bit: one 8-bit pass
    "bc256": (256, 100_000, 1 << 20, 5000, False),                   # 8 bits: one 8-bit pass
    "bc257": (257, 100_000, 1 << 20, 5000, False),                   # 9 bits: one 9-bit pass
    "bc513": (513, 150_000, 1 << 20, 5000, True),                    # 10 bits: group-by, hw 2
    "bc262144_packed": (262_144, 700_000, (1 << 23) - 1, 5000, True),  # 18 bits: group-by, hw 9, 23-bit tokens: bit 31 used
    "bc262144_wide": (262_144, 700_000, 1 << 23, 5000, False),        # one more token bit: 2 x 9 pair sort
    "bc262144_unk": (262_144, 700_000, 1000, (1 << 23) - 1, True),   # the unk id alone sets the 23-bit token width
    "bc262144_unk_wide": (262_144, 700_000, 1000, 1 << 23, False),   # ... and one more bit of it: pair sort
    "bc262145": (262_145, 700_000, 1 << 20, 5000, False),            # 19 bits: 3 x 8 pair sort
    "bc2p25": ((1 << 25) + 1, 1_000_000, 1 << 20, 5000, False),       # 26 bits: 3 x 9 pair sort
}


@pytest.fixture(scope="module")
def frag_data(env):
    """Per case (built on first use): the device and oracle indexes, the fragments and the oracle's tokenization."""
    cache = {}

    def get(case):
        if case not in cache:
            n_bc, n, max_val, unk, _ = FRAG_CASES[case]
            rng = np.random.default_rng(zlib.crc32(f"frag/{case}".encode()))
            g, o = _universe(env, rng, 5000, max_val)
            q = _fragments(rng, n, n_bc)
            cache[case] = types.SimpleNamespace(g=g, q=q, n_bc=n_bc, unk=unk, ref=o.tokenize_fragments(*q, n_bc, unk))
        return cache[case]
    return get


def _check_host(d):
    off, ids = d.g.tokenize_fragments(*d.q, d.n_bc, d.unk)
    assert np.array_equal(off, d.ref[0])
    assert np.array_equal(ids, d.ref[1])


def _check_dev(env, d, lead=0):
    """gtgpu_tokenize_fragments_dev with d_out_ids `lead` elements into a buffer (an odd lead misaligns it)."""
    import torch
    t = [torch.from_numpy(a.view(np.int32)).to("cuda") for a in d.q]
    total = int(d.ref[0][-1])
    cap = total + 17
    d_ids = _empty(cap, lead)
    d_bco, d_total = _empty(d.n_bc + 1, wide=True), _empty(1, wide=True)
    torch.cuda.synchronize()
    d.g.tokenize_fragments_dev(len(d.q[0]), *(x.data_ptr() for x in t), d.n_bc, d.unk, d_bco.data_ptr(), _ptr(d_ids, lead), cap,
                               d_total.data_ptr())
    env.stream.synchronize()
    assert int(_host(d_total)[0]) == total
    assert np.array_equal(_host(d_bco)[:d.n_bc + 1], d.ref[0])
    ids = _host(d_ids)
    assert np.array_equal(ids[lead:lead + total], d.ref[1])
    assert (ids[:lead] == SENT32).all() and (ids[lead + cap:] == SENT32).all()


def _pair_sort_cases():
    return [(c, s) for c, v in FRAG_CASES.items() for s in ((0,) if v[4] else (0, 1, 2))]


@pytest.mark.parametrize("case,shape", _pair_sort_cases())
def test_fragments_every_plan(env, shim, frag_data, monkeypatch, case, shape):
    """tokenize_fragments and tokenize_fragments_dev against the oracle at every plan the barcode sort can take: one pass of
    8 or 9 bits, the packed group-by on both sides of its 32-bit boundary (set by index vals or by unk_id), three passes of
    8 and of 9 bits; the pair-sort plans under every scatter tile shape."""
    n_bc, _, max_val, unk, group = FRAG_CASES[case]
    assert bool(shim.shim_radix_group_fits(n_bc, max(max_val, unk))) == group  # the case takes the path it names
    monkeypatch.setenv("GTGPU_RS_SHAPE", str(shape))
    d = frag_data(case)
    _check_host(d)
    _check_dev(env, d)


@pytest.mark.parametrize("case", [c for c, v in FRAG_CASES.items() if v[4]])
def test_fragments_pair_sort_equals_group_by(env, frag_data, monkeypatch, case):
    """GTGPU_NO_GROUP_SORT=1 sends the packed group-by's cases to the pair sort: same result."""
    monkeypatch.setenv("GTGPU_NO_GROUP_SORT", "1")
    d = frag_data(case)
    _check_host(d)
    _check_dev(env, d)


@pytest.mark.parametrize("case", ["bc262144_packed", "bc262144_wide", "bc262145"])
def test_fragments_dev_misaligned_ids(env, frag_data, case):
    """d_out_ids at an odd element offset: with an even pass count it is the sort's first input (staged by 4-byte copies),
    with an odd one the input of the middle pass."""
    _check_dev(env, frag_data(case), lead=1)


@pytest.mark.parametrize("max_val", [255, 256, 511, (1 << 17) - 1, 1 << 17])
@pytest.mark.parametrize("n_bc", [1, 513, 262_145])
def test_score_barcodes_plans(env, n_bc, max_val):
    """score_barcodes sorts (peak, barcode) pairs by peak id, then by barcode: peak-id widths of 8, 9, 17 and 18 bits
    against barcode counts of 1, 10 and 19 bits."""
    from oracle import oracle as orc
    rng = np.random.default_rng(zlib.crc32(f"score/{n_bc}/{max_val}".encode()))
    g, o = _universe(env, rng, 20_000, max_val)
    qc, qs, qe, bc = _fragments(rng, 200_000, n_bc)
    got, ref = g.score_barcodes(qc, qs, qe, bc, n_bc), orc.score_barcodes(o, qc, qs, qe, bc, n_bc)
    for a, b in zip(got, ref):
        assert np.array_equal(a, b)
    assert int(got[1].max()) == max_val


def test_parse_bed_sort_full_u32_range(env):
    """gtgpu_parse_bed's stable (name, start) sort with starts over the whole u32 range (at and above 2^31, 4 294 967 295,
    heavy ties) and 300 names, so the name-rank pass has 9-bit digits; reference: numpy lexsort on (start, name rank)."""
    from gtars_b200 import ffi
    rng = np.random.default_rng(31)
    names = [f"chr{i}_{''.join(rng.choice(list('acgtxyz'), 5))}" for i in range(300)]
    table = [names[i] for i in rng.permutation(len(names))]   # ids in this order; the sort uses the names' string order
    n = 200_000
    name_of = rng.integers(0, len(names), n)
    start = rng.integers(0, 1 << 32, n, dtype=np.uint64)
    k = rng.random(n)
    start = np.where(k < 0.3, rng.integers(1 << 31, 1 << 32, n, dtype=np.uint64), start)
    start = np.where((k >= 0.3) & (k < 0.4), np.uint64(0xFFFFFFFF), start)
    start = np.where((k >= 0.4) & (k < 0.6), rng.choice(np.array([0, 7, 1 << 31, 0x80000001], np.uint64), n), start)
    end = np.minimum(start + rng.integers(0, 1000, n).astype(np.uint64), 0xFFFFFFFF)
    text = "".join(f"{names[c]}\t{s}\t{e}\n" for c, s, e in zip(name_of.tolist(), start.tolist(), end.tolist())).encode()
    blob, offs = ffi._names_blob(table)
    n_out = C.c_uint64(0)
    h = [C.c_void_p() for _ in range(3)]
    ffi.check(ffi.lib().gtgpu_parse_bed(env.ctx._h, text, len(text), len(table), blob, ffi._p(offs), C.byref(n_out),
                                        *(C.byref(x) for x in h)))
    c, s, e = (ffi._take(x) for x in h)
    lex_rank = np.empty(len(names), np.int64)
    lex_rank[np.argsort(np.array(names))] = np.arange(len(names))
    table_id = np.array([table.index(nm) for nm in names], np.uint32)
    order = np.lexsort((start, lex_rank[name_of]))
    assert n_out.value == n
    assert np.array_equal(c, table_id[name_of][order])
    assert np.array_equal(s, start[order].astype(np.uint32))
    assert np.array_equal(e, end[order].astype(np.uint32))
