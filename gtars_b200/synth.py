"""Counter-based synthetic hg38-shaped workloads (SURVEY.md §8d) — torch tensors on any device.

Every value is a pure function of (seed, stream, index) through splitmix64, so any shard of any workload can be
regenerated independently (per file, per rank) and host and device copies are identical.
Coordinates stay below 2^31, so int32 storage is bit-identical to the uint32 the C ABI takes.
"""
from __future__ import annotations

import torch

HG38 = [("chr1", 248956422), ("chr2", 242193529), ("chr3", 198295559), ("chr4", 190214555), ("chr5", 181538259),
        ("chr6", 170805979), ("chr7", 159345973), ("chr8", 145138636), ("chr9", 138394717), ("chr10", 133797422),
        ("chr11", 135086622), ("chr12", 133275309), ("chr13", 114364328), ("chr14", 107043718), ("chr15", 101991189),
        ("chr16", 90338345), ("chr17", 83257441), ("chr18", 80373285), ("chr19", 58617616), ("chr20", 64444167),
        ("chr21", 46709983), ("chr22", 50818468), ("chrX", 156040895), ("chrY", 57227415), ("chrM", 16569)]
CHROM_NAMES = [n for n, _ in HG38]
CHROM_SIZES = [s for _, s in HG38]
N_CHROMS = len(HG38)
GENOME = sum(CHROM_SIZES)

SEED_UNIVERSE, SEED_QUERIES, SEED_FRAGMENTS, SEED_LOLA_DB, SEED_LOLA_USER = (0x5EED0001, 0x5EED0002, 0x5EED0003,
                                                                             0x5EED0004, 0x5EED0005)
_M63 = (1 << 63) - 1


def _i64(v: int) -> int:
    v &= (1 << 64) - 1
    return v - (1 << 64) if v >= (1 << 63) else v


def _lsr(x: torch.Tensor, k: int) -> torch.Tensor:
    return (x >> k) & ((1 << (64 - k)) - 1)


def splitmix64(x: torch.Tensor) -> torch.Tensor:
    """splitmix64 finaliser on int64 tensors (two's-complement wrap == uint64 arithmetic)."""
    x = x + _i64(0x9E3779B97F4A7C15)
    x = (x ^ _lsr(x, 30)) * _i64(0xBF58476D1CE4E5B9)
    x = (x ^ _lsr(x, 27)) * _i64(0x94D049BB133111EB)
    return x ^ _lsr(x, 31)


def rand_u63(seed: int, stream: int, index: torch.Tensor) -> torch.Tensor:
    """Non-negative 63-bit draw for each counter value."""
    return splitmix64(index + _i64(seed ^ (stream << 56))) & _M63


def lex_rank(device) -> torch.Tensor:
    """rank of each dense chromosome id under Rust's String ordering (RegionSet::sort, region_set.rs:502-505)."""
    order = sorted(range(N_CHROMS), key=lambda i: CHROM_NAMES[i])
    r = torch.empty(N_CHROMS, dtype=torch.int64)
    for rank, i in enumerate(order):
        r[i] = rank
    return r.to(device)


def make_universe(n: int = 1_000_000, seed: int = SEED_UNIVERSE, device="cpu", nested_frac: float = 0.0) -> dict:
    """Consensus-peak-like universe: per chromosome n_c ∝ size non-overlapping peaks (one per equal slot), width
    150–1000 bp, written in a shuffled file order so token id != sorted rank.  nested_frac > 0 adds that fraction of
    wide intervals (10–500 kb) to force multi-hit queries and several AIList components (the C2n variant).

    Returns file-order tensors chr/start/end (int32) plus the chromosome-grouped arrays gtgpu_index_build takes
    (chrom_offsets int64, starts, ends, vals=file-order token id)."""
    dev = torch.device(device)
    sizes = torch.tensor(CHROM_SIZES, dtype=torch.int64)
    per = torch.clamp((sizes * n) // GENOME, min=1)
    per[0] += n - int(per.sum())  # rounding remainder goes to chr1
    chr_l, st_l, en_l = [], [], []
    base = 0
    for c in range(N_CHROMS):
        k = int(per[c])
        idx = torch.arange(base, base + k, dtype=torch.int64, device=dev)
        slot = CHROM_SIZES[c] // k
        width = 150 + rand_u63(seed, 1, idx) % 851
        width = torch.clamp(width, max=max(slot - 2, 1))
        room = torch.clamp(slot - width - 1, min=1)
        start = torch.arange(k, dtype=torch.int64, device=dev) * slot + rand_u63(seed, 2, idx) % room
        end = torch.clamp(start + width, max=CHROM_SIZES[c])
        chr_l.append(torch.full((k,), c, dtype=torch.int64, device=dev))
        st_l.append(start)
        en_l.append(end)
        base += k
    n_wide = int(n * nested_frac)
    if n_wide:
        idx = torch.arange(n_wide, dtype=torch.int64, device=dev)
        c, pos = _genome_pos(rand_u63(seed, 3, idx), dev)
        width = 10_000 + rand_u63(seed, 4, idx) % 490_001
        csz = torch.tensor(CHROM_SIZES, dtype=torch.int64, device=dev)[c]
        chr_l.append(c)
        st_l.append(pos)
        en_l.append(torch.minimum(pos + width, csz))
    chr_s, st_s, en_s = torch.cat(chr_l), torch.cat(st_l), torch.cat(en_l)
    total = chr_s.numel()
    # shuffled file order
    perm = torch.argsort(rand_u63(seed, 5, torch.arange(total, dtype=torch.int64, device=dev)))
    chr_f, st_f, en_f = chr_s[perm], st_s[perm], en_s[perm]
    # chromosome-grouped, file order kept inside a chromosome (what Tokenizer's core builder sees)
    grp = torch.sort(chr_f, stable=True).indices
    counts = torch.bincount(chr_f, minlength=N_CHROMS)
    offs = torch.zeros(N_CHROMS + 1, dtype=torch.int64, device=dev)
    offs[1:] = torch.cumsum(counts, 0)
    return dict(n=total, chr=chr_f.int(), start=st_f.int(), end=en_f.int(), chrom_offsets=offs,
                g_start=st_f[grp].int(), g_end=en_f[grp].int(), g_val=grp.int(), unk_id=total)


def _genome_pos(u: torch.Tensor, dev):
    """Uniform 63-bit draws → (chromosome ∝ size, position) by inverting the cumulative chromosome lengths."""
    cum = torch.zeros(N_CHROMS + 1, dtype=torch.int64)
    cum[1:] = torch.cumsum(torch.tensor(CHROM_SIZES, dtype=torch.int64), 0)
    cum = cum.to(dev)
    g = u % GENOME
    c = torch.searchsorted(cum, g, right=True) - 1
    return c, g - cum[c]


def make_query_files(universe: dict, n_files: int, per_file: int, seed: int = SEED_QUERIES, device="cpu",
                     first_file: int = 0, sort_files: bool = True, unknown_frac_ppm: int = 0, width_scale: int = 1) -> dict:
    """BED-file-like query batches: 80 % a universe peak jittered ±100 bp, 20 % uniform background, width
    200–600 bp; each file sorted by (chromosome name, start) like RegionSet::try_from.  Files
    [first_file, first_file + n_files) of the infinite stream, so ranks can shard by file."""
    dev = torch.device(device)
    n = n_files * per_file
    idx = torch.arange(first_file * per_file, first_file * per_file + n, dtype=torch.int64, device=dev)
    kind = rand_u63(seed, 1, idx) % 5
    width = (200 + rand_u63(seed, 2, idx) % 401) * width_scale
    # peak-derived queries
    u_chr = universe["chr"].to(dev).long()
    u_start = universe["start"].to(dev).long()
    p = rand_u63(seed, 3, idx) % universe["n"]
    jitter = rand_u63(seed, 4, idx) % 201 - 100
    pk_chr = u_chr[p]
    pk_start = torch.clamp(u_start[p] + jitter, min=0)
    # background queries
    bg_chr, bg_start = _genome_pos(rand_u63(seed, 5, idx), dev)
    is_pk = kind < 4
    chr_ = torch.where(is_pk, pk_chr, bg_chr)
    start = torch.where(is_pk, pk_start, bg_start)
    csz = torch.tensor(CHROM_SIZES, dtype=torch.int64, device=dev)[chr_]
    start = torch.minimum(start, csz - 1)
    end = torch.minimum(start + width, csz)
    if sort_files:
        key = (lex_rank(dev)[chr_] << 32) | start
        order = torch.sort(key.view(n_files, per_file), dim=1, stable=True).indices
        order = (order + torch.arange(n_files, device=dev).view(-1, 1) * per_file).view(-1)
        chr_, start, end = chr_[order], start[order], end[order]
    if unknown_frac_ppm:
        unk = rand_u63(seed, 6, idx) % 1_000_000 < unknown_frac_ppm
        chr_ = torch.where(unk, torch.full_like(chr_, -1), chr_)  # -1 as int32 == 0xFFFFFFFF
    offs = torch.arange(n_files + 1, dtype=torch.int64, device=dev) * per_file
    return dict(n=n, chr=chr_.int(), start=start.int(), end=end.int(), file_offsets=offs)


def make_uniform_intervals(n: int, seed: int, device="cpu", min_w: int = 100, max_w: int = 10_000,
                           log_uniform: bool = True, first: int = 0) -> dict:
    """Uniform genome positions with (log-)uniform widths: the C3 database / query generator."""
    dev = torch.device(device)
    idx = torch.arange(first, first + n, dtype=torch.int64, device=dev)
    c, pos = _genome_pos(rand_u63(seed, 1, idx), dev)
    u = rand_u63(seed, 2, idx)
    if log_uniform:
        # integer-only log-uniform: uniform octave, uniform mantissa inside it (bit-identical on CPU and GPU)
        n_oct = max((max_w // min_w).bit_length(), 1)
        lo = min_w << (u % n_oct)
        width = torch.clamp(lo + _lsr(u, 8) % lo, max=max_w)
    else:
        width = min_w + u % (max_w - min_w + 1)
    csz = torch.tensor(CHROM_SIZES, dtype=torch.int64, device=dev)[c]
    pos = torch.minimum(pos, csz - 1)
    end = torch.minimum(pos + torch.clamp(width, min=1), csz)
    return dict(n=n, chr=c.int(), start=pos.int(), end=end.int())


def group_by_chrom(chr_: torch.Tensor, start: torch.Tensor, end: torch.Tensor) -> dict:
    """Insertion-order intervals → the chromosome-grouped arrays gtgpu_index_build takes (val = input index)."""
    grp = torch.sort(chr_.long(), stable=True).indices
    counts = torch.bincount(chr_.long(), minlength=N_CHROMS)
    offs = torch.zeros(N_CHROMS + 1, dtype=torch.int64, device=chr_.device)
    offs[1:] = torch.cumsum(counts, 0)
    return dict(chrom_offsets=offs, g_start=start[grp], g_end=end[grp], g_val=grp.int())


# ---- fragment files as text (numpy, for the text-ingest paths) ------------------------------------------------------------------
FRAGMENT_LINE = 40  # "chrNN" padded to 5 + TAB + 10-digit start + TAB + 10-digit end + TAB + "BC" + 7 digits + TAB + "1" + LF


def make_fragment_arrays(n: int, seed: int, n_barcodes: int):
    """Seeded fragments on the hg38-shaped chromosomes: (chr id into CHROM_NAMES, start, end, barcode number) as numpy
    uint32 arrays, 40 .. 1000 bp long."""
    import numpy as np
    rng = np.random.default_rng(seed)
    sizes = np.array(CHROM_SIZES, dtype=np.int64)
    c = rng.choice(len(sizes), n, p=sizes / sizes.sum()).astype(np.uint32)
    s = (rng.random(n) * (sizes[c] - 2000)).astype(np.uint32)
    e = s + rng.integers(40, 1000, n, dtype=np.uint32)
    b = rng.integers(0, n_barcodes, n, dtype=np.uint32)
    return c, s, e, b


def fragment_text(chr_id, start, end, barcode):
    """Vectorised fixed-width fragment lines as a uint8 array (FRAGMENT_LINE bytes each): the name padded with spaces (split
    on whitespace like any separator), start / end zero-padded (str::parse::<u32> accepts leading zeros), barcode "BC%07d",
    support 1.  barcode < 10^7."""
    import numpy as np
    tab = np.array([list(nm.ljust(5).encode()) for nm in CHROM_NAMES], dtype=np.uint8)
    out = np.empty((len(start), FRAGMENT_LINE), dtype=np.uint8)
    out[:, 0:5] = tab[chr_id]
    out[:, [5, 16, 27, 37]] = 9

    def digits(col, v, width):
        v = np.asarray(v).astype(np.uint64)
        for j in range(width - 1, -1, -1):
            out[:, col + j] = (v % 10).astype(np.uint8) + 48
            v //= 10

    digits(6, start, 10)
    digits(17, end, 10)
    out[:, 28:30] = np.frombuffer(b"BC", dtype=np.uint8)
    digits(30, barcode, 7)
    out[:, 38] = ord("1")
    out[:, 39] = 10
    return out.reshape(-1)
