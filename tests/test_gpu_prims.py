"""GPU suite: the multi-block primitives every ordered output rests on -- hc_scan::exclusive_u32, hc_radix::sort_pairs and
hc_line_index (hc_text.cuh) -- compared exactly with numpy through the test-only C entry points of
tests/cuda/hc_prims_shim.cu.  Each primitive has a second, carry-propagating loop in a single-block kernel that only runs
past a fixed size: more than 1024 block sums (scan_block_sums), more than 16384 sort tiles (the digit-matrix scan of
sort_pairs, 256 cells per tile) and more than 1024 text tiles (scan_counts).  The size lists below straddle those sizes;
test_cases_cross_their_boundaries (no GPU) checks that they still do."""
import ctypes
import os

import numpy as np
import pytest

# the sizes the primitives are built for (checked against the headers by test_shim_constants)
SCAN_THREADS, SCAN_PER_BLOCK = 1024, 4096             # hc_scan::THREADS, hc_scan::PER_BLOCK
RADIX_DIGITS, RADIX_TILE = 256, 2048                  # hc_radix::THREADS (= digit values), hc_radix::TILE
TEXT_TILE, COUNTS_BLOCK = 4096, 1024                  # newline TILE of hc_text.cuh, threads of scan_counts
SCAN_CARRY = SCAN_THREADS * SCAN_PER_BLOCK            # inputs above this: scan_block_sums carries between its passes
SORT_CARRY = SCAN_CARRY // RADIX_DIGITS * RADIX_TILE  # records above this: the digit-matrix scan carries
TEXT_CARRY = COUNTS_BLOCK * TEXT_TILE                 # text bytes above this: scan_counts carries

SCAN_SIZES = [0, 1, 4095, 4096, 4097, SCAN_CARRY - 1, SCAN_CARRY, SCAN_CARRY + 1, 4096 * 1025 + 17, 3 * SCAN_CARRY + 5]
SCAN_PATTERNS = ["random", "all_ones", "zero", "last_only"]
TEXT_SIZES = [1, 15, 16, 17, 4095, 4096, 4097, TEXT_CARRY - 1, TEXT_CARRY + 1, 4096 * 1025, 10_000_037]
TEXT_DENSITIES = ["none", "all", "random", "last_newline", "last_not_newline"]
SORT_SMALL = [1, 2, RADIX_TILE - 1, RADIX_TILE, RADIX_TILE + 1]
SORT_BIG = [SORT_CARRY, SORT_CARRY + 1]
SORT_PATTERNS = ["equal", "digit0", "digit7", "digit8", "digit15", "high_only", "reverse", "duplicates", "fno_keys"]
SORT_BIG_PATTERNS = ["equal", "digit8", "reverse", "duplicates", "fno_keys"]    # lexsort of 33 M records takes seconds

SENT64 = np.uint64(0xA5A5A5A5A5A5A5A5)
GUARD = 64                                            # sentinel entries behind every output buffer


def scan_blocks(n):
    return (n + SCAN_PER_BLOCK - 1) // SCAN_PER_BLOCK


def blocks_for(n):
    """hc_scan::blocks_for: what the library's callers allocate for d_bsum."""
    return scan_blocks(n) + 1


def sort_cells(n):
    return RADIX_DIGITS * ((n + RADIX_TILE - 1) // RADIX_TILE)


def text_tiles(n):
    return (n + TEXT_TILE - 1) // TEXT_TILE


def test_cases_cross_their_boundaries():
    """Each size list reaches past the size where its primitive's carry loop starts, and sits on both sides of it."""
    nb = [scan_blocks(n) for n in SCAN_SIZES]
    assert SCAN_THREADS in nb and SCAN_THREADS + 1 in nb and max(nb) > 3 * SCAN_THREADS       # exactly one pass, two, four
    assert 0 in nb and 1 in nb and 2 in nb
    assert any(n % SCAN_PER_BLOCK and scan_blocks(n) > SCAN_THREADS for n in SCAN_SIZES)     # partial last block
    cells = [scan_blocks(sort_cells(n)) for n in SORT_BIG]
    assert sort_cells(SORT_CARRY) == SCAN_CARRY and cells == [SCAN_THREADS, SCAN_THREADS + 1]
    assert [(n + RADIX_TILE - 1) // RADIX_TILE for n in SORT_SMALL] == [1, 1, 1, 1, 2]
    tiles = [text_tiles(n) for n in TEXT_SIZES]
    assert COUNTS_BLOCK in tiles and COUNTS_BLOCK + 1 in tiles and max(tiles) > 2 * COUNTS_BLOCK
    assert {n % 16 for n in TEXT_SIZES} >= {0, 1, 15}                                         # whole and partial 16-byte words


@pytest.fixture(scope="module")
def shim():
    from haploconduct_b200 import build as B, capi

    if os.path.exists(B.NVCC):
        B.build()
    assert os.path.exists(B.PRIMS_SHIM), "libhc_prims_shim.so missing: haploconduct_b200/build.py builds it"
    capi.lib()                                        # libhc_b200.so first: the shim resolves hc_scratch_alloc from it
    L = ctypes.CDLL(B.PRIMS_SHIM)
    P = ctypes.c_void_p
    u64 = ctypes.c_uint64
    L.hcp_constants.argtypes, L.hcp_constants.restype = [P], None
    L.hcp_blocks_for.argtypes, L.hcp_blocks_for.restype = [u64], u64
    L.hcp_exclusive_u32.argtypes, L.hcp_exclusive_u32.restype = [P, u64, P, u64, P, P, u64], ctypes.c_int
    L.hcp_sort_pairs.argtypes, L.hcp_sort_pairs.restype = [P, P, u64, P], ctypes.c_int
    L.hcp_line_index.argtypes, L.hcp_line_index.restype = [P, u64, u64, P, u64, P, P], ctypes.c_int
    return L


@pytest.mark.gpu
def test_shim_constants(shim):
    c = np.zeros(6, dtype=np.uint64)
    shim.hcp_constants(c.ctypes.data)
    assert c.tolist() == [SCAN_THREADS, SCAN_PER_BLOCK, RADIX_DIGITS, RADIX_TILE, TEXT_TILE, COUNTS_BLOCK]
    for n in SCAN_SIZES:
        assert shim.hcp_blocks_for(n) == blocks_for(n)


# ---- hc_scan::exclusive_u32 -------------------------------------------------------------------------------------------
def scan_input(n, pattern):
    if pattern == "random":
        return np.random.default_rng(n).integers(0, 2 ** 32, n, dtype=np.uint32)
    if pattern == "all_ones":
        return np.full(n, 0xffffffff, dtype=np.uint32)
    x = np.zeros(n, dtype=np.uint32)
    if pattern == "last_only" and n:
        x[-1] = 0xfffffffe
    return x


@pytest.mark.gpu
@pytest.mark.parametrize("pattern", SCAN_PATTERNS)
@pytest.mark.parametrize("n", SCAN_SIZES)
def test_exclusive_u32(shim, n, pattern):
    x = scan_input(n, pattern)
    inc = np.cumsum(x, dtype=np.uint64)
    want = np.concatenate([np.zeros(1, np.uint64), inc[:-1]]) if n else np.zeros(0, np.uint64)
    want_total = int(inc[-1]) if n else 0
    nb = blocks_for(n)                                # exactly what the library allocates, then the guard
    out = np.full(n + GUARD, SENT64, dtype=np.uint64)
    bsum = np.full(nb + GUARD, SENT64, dtype=np.uint64)
    total = np.full(1, SENT64, dtype=np.uint64)
    rc = shim.hcp_exclusive_u32(x.ctypes.data, n, out.ctypes.data, len(out), total.ctypes.data, bsum.ctypes.data, len(bsum))
    assert rc == 0
    assert int(total[0]) == want_total
    assert np.array_equal(out[:n], want), "first difference at %s" % np.flatnonzero(out[:n] != want)[:5]
    assert (out[n:] == SENT64).all(), "written past out[n)"
    assert (bsum[nb:] == SENT64).all(), "written past d_bsum[blocks_for(n))"
    used = scan_blocks(n)                             # after the scan of the block sums: every block's offset
    assert np.array_equal(bsum[:used], want[::SCAN_PER_BLOCK])
    if pattern == "all_ones" and n > 2:
        assert want_total >= 2 ** 32


# ---- hc_line_index --------------------------------------------------------------------------------------------------
def text_of(n, density):
    rng = np.random.default_rng(1000 + n)
    t = rng.integers(32, 127, n, dtype=np.uint8)      # printable, never '\n'
    if density == "all":
        t[:] = 10
    elif density == "random":
        t[rng.random(n) < 0.05] = 10
    elif density == "last_newline":
        t[rng.random(n) < 0.01] = 10
        t[-1] = 10
    elif density == "last_not_newline":
        t[rng.random(n) < 0.01] = 10
        t[-1] = ord("A")
    return t


@pytest.mark.gpu
@pytest.mark.parametrize("density", TEXT_DENSITIES)
@pytest.mark.parametrize("n", TEXT_SIZES)
def test_line_index(shim, n, density):
    """Every text at byte offsets 0..15 from a 16-byte boundary: nl_mask16 reads aligned text 16 bytes at a time and
    unaligned text byte by byte."""
    t = text_of(n, density)
    want = np.concatenate([np.zeros(1, np.uint64), (np.flatnonzero(t == 10) + 1).astype(np.uint64)])
    want_lines = len(want) - 1 + int(t[-1] != 10)
    if density == "none":
        assert len(want) == 1
    if density == "all":
        assert len(want) == n + 1
    for off in range(16):
        ls = np.full(len(want) + GUARD, SENT64, dtype=np.uint64)
        nl, lines = ctypes.c_uint64(0), ctypes.c_uint64(0)
        rc = shim.hcp_line_index(t.ctypes.data, n, off, ls.ctypes.data, len(ls), ctypes.byref(nl), ctypes.byref(lines))
        assert rc == 0, off
        assert (nl.value, lines.value) == (len(want) - 1, want_lines), off
        assert np.array_equal(ls[:len(want)], want), (off, np.flatnonzero(ls[:len(want)] != want)[:5])
        assert (ls[len(want):] == SENT64).all(), off


# ---- hc_radix::sort_pairs -------------------------------------------------------------------------------------------
def dec_key(v):
    """K(v) of hc_fno_text.cu: v zero-padded to ten digits, times ten, plus (digits - 1)."""
    v = np.asarray(v, dtype=np.uint64)
    d = np.ones(len(v), dtype=np.uint64)
    for p in range(1, 10):
        d += (v >= np.uint64(10 ** p)).astype(np.uint64)
    return v * (np.uint64(10) ** (np.uint64(10) - d)) * np.uint64(10) + (d - np.uint64(1))


def sort_keys(n, pattern):
    """(low 64 bits, high 64 bits) of n keys."""
    rng = np.random.default_rng(7 * n + len(pattern))
    base_lo, base_hi = np.uint64(0x0123456789ABCDEF), np.uint64(0xFEDCBA9876543210)
    lo, hi = np.full(n, base_lo, np.uint64), np.full(n, base_hi, np.uint64)
    if pattern.startswith("digit"):                   # keys differ in that one digit only (a few values, many equal)
        p = int(pattern[5:])
        d = rng.integers(0, 256, n, dtype=np.uint64) if n > 512 else rng.integers(0, 3, n, dtype=np.uint64)
        d[:2] = [2, 1][:n]                            # the digit varies whenever there are two keys
        half, sh = (lo, hi)[p // 8], np.uint64(8 * (p % 8))
        half &= ~(np.uint64(0xff) << sh)
        half |= d << sh
    elif pattern == "high_only":
        hi = rng.integers(0, 2 ** 63, n, dtype=np.uint64) * np.uint64(2) + rng.integers(0, 2, n, dtype=np.uint64)
        hi[::3] = hi[0]
    elif pattern == "reverse":
        r = np.arange(n, dtype=np.uint64)[::-1].copy()
        hi = r * np.uint64(0x10001)
        lo = r * np.uint64(0x9E3779B97F4A7C15)
    elif pattern == "duplicates":                     # 37 distinct keys, every digit position varies
        pool_lo = rng.integers(0, 2 ** 64, 37, dtype=np.uint64)
        pool_hi = rng.integers(0, 2 ** 64, 37, dtype=np.uint64)
        pick = rng.integers(0, 37, n)
        lo, hi = pool_lo[pick], pool_hi[pick]
    elif pattern == "fno_keys":                       # (K(id2), K(id1)) of ids of every digit count, shared prefixes
        pool = np.array([0, 1, 2, 9, 10, 11, 19, 100, 1000000000, 4294967294, 4294967295] +
                        [int(x) for d in range(1, 11) for x in rng.integers(10 ** (d - 1), min(10 ** d, 2 ** 32), 6)], dtype=np.uint64)
        lo = dec_key(pool[rng.integers(0, len(pool), n)])
        hi = dec_key(pool[rng.integers(0, len(pool), n)])
    else:
        assert pattern == "equal"
    return lo, hi


def varying_digits(lo, hi):
    diff = [np.bitwise_and.reduce(h) ^ np.bitwise_or.reduce(h) for h in (lo, hi)] if len(lo) else [np.uint64(0)] * 2
    return sum(1 for p in range(16) if (int(diff[p // 8]) >> (8 * (p % 8))) & 0xff)


def check_sort(shim, n, pattern):
    lo, hi = sort_keys(n, pattern)
    keys = np.empty((n, 2), dtype=np.uint64)
    keys[:, 0], keys[:, 1] = lo, hi
    vals = np.arange(n, dtype=np.uint32)              # value = input index: stability is checked directly
    # np.lexsort is stable, so equal keys keep index order, as lexsort((index, lo, hi)) would have them
    want = np.lexsort((lo, hi))
    in_tmp = ctypes.c_int(-2)
    assert shim.hcp_sort_pairs(keys.ctypes.data, vals.ctypes.data, n, ctypes.byref(in_tmp)) == 0
    passes = varying_digits(lo, hi)
    if pattern == "equal":
        assert passes == 0                            # every digit skipped: the input buffers are the result
    elif pattern.startswith("digit"):
        assert passes == (1 if n > 1 else 0)
    elif pattern == "reverse":
        assert np.array_equal(want, np.arange(n)[::-1])
    elif pattern in ("duplicates", "reverse") and n > 2 ** 20:
        assert passes >= 8
    assert in_tmp.value == passes % 2, "result buffer: %d passes, in_tmp %d" % (passes, in_tmp.value)
    assert np.array_equal(vals, want), "first difference at %s" % np.flatnonzero(vals != want)[:5]
    assert np.array_equal(keys[:, 0], lo[want]) and np.array_equal(keys[:, 1], hi[want])


@pytest.mark.gpu
@pytest.mark.parametrize("pattern", SORT_PATTERNS)
@pytest.mark.parametrize("n", SORT_SMALL)
def test_sort_pairs(shim, n, pattern):
    check_sort(shim, n, pattern)


@pytest.mark.gpu
@pytest.mark.parametrize("pattern", SORT_BIG_PATTERNS)
@pytest.mark.parametrize("n", SORT_BIG)
def test_sort_pairs_past_the_cell_scan(shim, n, pattern):
    """16384 tiles are 4,194,304 digit-matrix cells, one full pass of scan_block_sums; one record more needs a second."""
    assert scan_blocks(sort_cells(n)) >= SCAN_THREADS
    check_sort(shim, n, pattern)
