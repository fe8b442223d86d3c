"""GPU tests: the sorted-key primitives (csrc/sort_scan.cu) bit for bit against their exact references
(tests/sort_scan_reference.py), through the parity hooks b200ppf_debug_*.

The inputs are seeded and chosen where the kernels change path or carry state from one block to the next:
  radix sort     512- and 4096-element tiles (the switch at T = 4 * SMs * 4096 elements), one and several column-scan
                 chunks of 256 tiles, partial last tiles, one to four 8-bit passes (the pass count follows the largest
                 key), key distributions that fill one digit run per tile or leave digits empty, every payload
                 combination the sort dispatches, and stability through the payloads;
  lower_bounds   shifts of the phase-cell keys, keys past n_keys << shift, a list length read from the device, a target
                 k << shift of 2^32;
  flag_scan      one block, more than 1024 block sums (the scan of the block sums carries from one 1024 chunk to the
                 next), flag words other than 0 and 1;
  scan_rows      rows of one to several 1024-word chunks, up to 64 rows;
  run_heads      a run boundary on a block edge.
Outputs are handed to the device with canary words behind the documented range: those must come back untouched.
"""
import functools

import numpy as np
import pytest

import sort_scan_reference as ref

pytestmark = pytest.mark.gpu

CANARY = 0xA5A5A5A5
TILE_SMALL, TILE_BIG, SCAN_CHUNK = 512, 4096, 256


@functools.lru_cache(None)
def _big_tile_threshold():
    """T: the sort takes 4096-element tiles from T elements on"""
    import torch
    return 4 * torch.cuda.get_device_properties(0).multi_processor_count * TILE_BIG


def _big_chunk_edge():
    """the first multiple of a 4096-element-tile column-scan chunk at or above T"""
    chunk = SCAN_CHUNK * TILE_BIG
    return -(-_big_tile_threshold() // chunk) * chunk


def _size(spec):
    """an element count, or (name, delta) of a count that depends on the SM count"""
    if isinstance(spec, int):
        return spec
    return {"T": _big_tile_threshold(), "big_chunk": _big_chunk_edge()}[spec[0]] + spec[1]


def _size_id(spec):
    return str(spec) if isinstance(spec, int) else f"{spec[0]}{spec[1]:+d}"


def _same(got, want, what):
    got, want = np.asarray(got), np.asarray(want)
    assert got.shape == want.shape, (what, got.shape, want.shape)
    bad = np.flatnonzero(got != want)
    assert bad.size == 0, f"{what}: {bad.size} words differ, first at {bad[0]}: {got[bad[0]]} != {want[bad[0]]}"


def _launches(ctx, call):
    before = ctx.launch_count
    out = call()
    return out, ctx.launch_count - before


# ---- radix sort ------------------------------------------------------------------------------------------------------

def _check_sort(ctx, keys, max_key, v0=None, v1=None, v0_iota=False):
    got, launches = _launches(ctx, lambda: ctx.debug_radix_sort(keys, max_key, v0, v1, v0_iota))
    want = ref.radix_sort(keys, max_key, v0, v1, v0_iota)
    for g, w, what in zip(got[:3], want[:3], ("keys", "v0", "v1")):
        assert (g is None) == (w is None), what
        if w is not None:
            _same(g, w, f"{what} (n {keys.size}, max_key {max_key})")
    assert got[3] == want[3], "result_in_alt is not the parity of the pass count"
    assert launches == (5 * ref.radix_passes(max_key) if keys.size else 0)


def _keys(rng, n, max_key, dist):
    """n keys in [0, max_key] (max_key clamped to 32 bits), max_key itself among them"""
    hi = min(max_key, ref.U32_MAX)
    uniform = rng.integers(0, hi + 1, n, dtype=np.uint64).astype(np.uint32)
    uniform[rng.integers(n)] = hi
    if dist == "uniform":
        return uniform
    if dist == "all_equal":
        return np.full(n, hi, np.uint32)
    if dist == "two_values":
        return np.where(rng.random(n) < 0.5, hi // 3, hi).astype(np.uint32)
    if dist == "sorted":
        return np.sort(uniform)
    if dist == "reversed":
        return np.sort(uniform)[::-1].copy()
    if dist == "const_low_byte":  # the low digit pass has one non-empty digit, the others many empty ones
        k = (rng.integers(0, (hi >> 8) + 1, n, dtype=np.uint64).astype(np.uint32) << np.uint32(8)) | np.uint32(hi & 0xFF)
        k[rng.integers(n)] = hi
        return k
    if dist == "dup_spread":  # a handful of values, each spread over every tile
        return rng.choice(np.append(rng.integers(0, hi + 1, 5, dtype=np.uint64), hi).astype(np.uint32), n)
    raise ValueError(dist)


def _garbage(rng, n):
    return rng.integers(0, 2 ** 32, n, dtype=np.uint32)


SORT_SIZES = [1, 31, 32, 33, 511, 512, 513, 4095, 4096, 4097,
              SCAN_CHUNK * TILE_SMALL - 1, SCAN_CHUNK * TILE_SMALL + 1,  # one / two column-scan chunks of small tiles
              ("T", -1), ("T", 0),                                       # the largest small-tile and smallest big-tile sort
              ("big_chunk", -1), ("big_chunk", 1),                       # a column-scan chunk boundary of big tiles
              2 ** 25 + 7]


@pytest.mark.parametrize("size", SORT_SIZES, ids=_size_id)
def test_radix_sort_sizes(ctx, size):
    n = _size(size)
    if isinstance(size, tuple) and size[0] == "big_chunk":
        assert n >= _big_tile_threshold()
    rng = np.random.default_rng(n)
    keys = _keys(rng, n, ref.U32_MAX, "uniform")
    _check_sort(ctx, keys, ref.U32_MAX, v0=_garbage(rng, n), v1=_garbage(rng, n), v0_iota=True)
    if n < 2 ** 25:  # three passes, the result in the alternate buffers; few distinct keys for stability
        _check_sort(ctx, _keys(rng, n, 2 ** 16, "dup_spread"), 2 ** 16, v0=_garbage(rng, n), v1=_garbage(rng, n))


MAX_KEYS = [0, 1, 255, 256, 2 ** 16 - 1, 2 ** 16, 2 ** 24 - 1, 2 ** 24, 2 ** 32 - 1, 2 ** 40]
DISTS = ["uniform", "all_equal", "two_values", "sorted", "reversed", "const_low_byte", "dup_spread"]


@pytest.mark.parametrize("dist", DISTS)
@pytest.mark.parametrize("max_key", MAX_KEYS)
def test_radix_sort_key_range_and_distribution(ctx, max_key, dist):
    """small tiles over two column-scan chunks and a partial last tile; v0 as iota carries each key's input position, so
    the order of equal keys is checked everywhere (max_key 0: the only pass is the one that writes the iota)"""
    n = SCAN_CHUNK * TILE_SMALL + 777
    rng = np.random.default_rng([max_key % 1000003, DISTS.index(dist)])
    _check_sort(ctx, _keys(rng, n, max_key, dist), max_key, v0=_garbage(rng, n), v1=_garbage(rng, n), v0_iota=True)


@pytest.mark.parametrize("dist", DISTS)
def test_radix_sort_big_tiles_distribution(ctx, dist):
    n = _big_tile_threshold() + 4097
    rng = np.random.default_rng([7, DISTS.index(dist)])
    _check_sort(ctx, _keys(rng, n, 2 ** 24, dist), 2 ** 24, v0=_garbage(rng, n), v0_iota=True)


PAYLOADS = {"none": (False, False, False), "v0": (True, False, False), "v0_iota": (True, True, False),
            "v1": (False, False, True), "v0_v1": (True, False, True), "v0_iota_v1": (True, True, True)}


@pytest.mark.parametrize("tile", ["small", "big"])
@pytest.mark.parametrize("mode", list(PAYLOADS))
def test_radix_sort_payload_modes(ctx, mode, tile):
    """every scatter instantiation: six payload combinations at both tile sizes, at one, three and four passes"""
    has_v0, iota, has_v1 = PAYLOADS[mode]
    n = 5 * TILE_SMALL + 100 if tile == "small" else _big_tile_threshold()
    rng = np.random.default_rng([n, list(PAYLOADS).index(mode)])
    for max_key in (0, 2 ** 16, ref.U32_MAX):
        keys = _keys(rng, n, max_key, "dup_spread")
        _check_sort(ctx, keys, max_key, v0=_garbage(rng, n) if has_v0 else None, v1=_garbage(rng, n) if has_v1 else None,
                    v0_iota=iota)


def test_radix_sort_of_nothing(ctx):
    got, launches = _launches(ctx, lambda: ctx.debug_radix_sort(np.zeros(0, np.uint32), ref.U32_MAX, v0=np.zeros(0),
                                                                v0_iota=True))
    assert got[0].size == 0 and got[1].size == 0 and got[3] is False and launches == 0


# ---- lower_bounds ----------------------------------------------------------------------------------------------------

def _check_lower_bounds(ctx, s, n_keys, shift, dev_len=None):
    canary = np.full(n_keys + 1 + 33, CANARY, np.uint32)
    got, launches = _launches(ctx, lambda: ctx.debug_lower_bounds(s, n_keys, shift, dev_len=dev_len, offsets=canary))
    _same(got[:n_keys + 1], ref.lower_bounds(s, n_keys, shift, dev_len), f"offsets (n_keys {n_keys}, shift {shift}, len {dev_len})")
    _same(got[n_keys + 1:], canary[n_keys + 1:], "words past offsets[n_keys]")
    assert launches == 1
    return got


def _sorted_keys(rng, n, n_keys, shift):
    """bucket starts, keys inside buckets, keys past n_keys << shift and a 0xFFFFFFFF end key (verification's)"""
    top = min((n_keys + 2) << shift, 2 ** 32)
    k = rng.integers(0, top, n, dtype=np.uint64)
    k[: n // 8] = rng.integers(0, n_keys + 1, n // 8).astype(np.uint64) << np.uint64(shift)
    k = np.sort(np.minimum(k, ref.U32_MAX)).astype(np.uint32)
    k[-1] = ref.U32_MAX
    return k


@pytest.mark.parametrize("shift", [0, 1, 4, 5, 9, 12, 20])
def test_lower_bounds(ctx, shift):
    rng = np.random.default_rng(shift)
    for n, n_keys in ((1, 1), (777, 40), (100_003, 3000), (1_000_000, 255)):
        s = _sorted_keys(rng, n, n_keys, shift)
        full = _check_lower_bounds(ctx, s, n_keys, shift)
        assert full[n_keys] < n  # points at the keys past the range, not at n
        for dev_len in (n, n // 3, 0):  # K4's compacted lists; 0 = its empty leaders list
            _check_lower_bounds(ctx, s, n_keys, shift, dev_len)
    _check_lower_bounds(ctx, np.zeros(0, np.uint32), 9, shift)


def test_lower_bounds_target_reaching_2_32(ctx):
    """k << shift == 2^32 is past every 32-bit key: offsets[n_keys] is the list length, not 0"""
    rng = np.random.default_rng(11)
    for n_keys, shift in ((256, 24), (2, 31), (16, 28), (4096, 20)):
        s = np.sort(rng.integers(0, 2 ** 32, 5000, dtype=np.uint64)).astype(np.uint32)
        s[-1] = ref.U32_MAX
        assert n_keys << shift == 2 ** 32
        assert _check_lower_bounds(ctx, s, n_keys, shift)[n_keys] == s.size
        assert _check_lower_bounds(ctx, s, n_keys, shift, dev_len=1234)[n_keys] == 1234


# ---- flag_scan -------------------------------------------------------------------------------------------------------

NOT_ONE = np.array([0, 2, 3, 0xFFFFFFFF], np.uint32)


def _flags(rng, n, density):
    if density == "zero":
        return np.zeros(n, np.uint32)
    if density == "one":
        return np.ones(n, np.uint32)
    if density == "alternating":
        return (np.arange(n) % 2 == 0).astype(np.uint32)
    if density in ("first", "last"):
        f = np.zeros(n, np.uint32)
        f[0 if density == "first" else n - 1] = 1
        return f
    if density == "not_one":  # words that are set but not 1: none counts
        return rng.choice(NOT_ONE[1:], n)
    p = {"random": 0.5, "sparse": 1e-3}[density]
    return np.where(rng.random(n) < p, np.uint32(1), rng.choice(NOT_ONE, n)).astype(np.uint32)


FLAG_SIZES = [1, 1023, 1024, 1025, 2 ** 20 - 1, 2 ** 20, 2 ** 20 + 1]  # 2^20: exactly 1024 block sums
DENSITIES = ["zero", "one", "alternating", "random", "sparse", "first", "last", "not_one"]
FLAG_CASES = [(n, d) for n in FLAG_SIZES for d in DENSITIES] + [(2 ** 26 + 5, d) for d in ("random", "last")]


@pytest.mark.parametrize("n,density", FLAG_CASES)
def test_flag_scan(ctx, n, density):
    rng = np.random.default_rng([n, DENSITIES.index(density)])
    flags = _flags(rng, n, density)
    want_rank, want_total = ref.flag_scan(flags)
    canary = np.full(n + 16, CANARY, np.uint32)
    for host_total in (False, True):
        (rank, total), launches = _launches(ctx, lambda: ctx.debug_flag_scan(flags, rank=canary, host_total=host_total,
                                                                             total=0x5A5A5A5A))
        _same(rank[:n], want_rank, f"rank (host total {host_total})")
        _same(rank[n:], canary[n:], "words past rank[n - 1]")
        assert total == want_total and launches == 3, (host_total, total, want_total, launches)


def test_flag_scan_of_nothing(ctx):
    canary = np.full(16, CANARY, np.uint32)
    for host_total in (False, True):
        (rank, total), launches = _launches(ctx, lambda: ctx.debug_flag_scan(np.zeros(0, np.uint32), rank=canary,
                                                                             host_total=host_total, total=0x5A5A5A5A))
        assert total == 0 and launches == 0
        _same(rank, canary, "rank of an empty scan")


# ---- scan_rows -------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("row_len", [0, 1, 31, 1023, 1024, 1025, 3 * 1024, 5000])
@pytest.mark.parametrize("n_rows", [1, 2, 7, 64])
def test_scan_rows(ctx, n_rows, row_len):
    """counts up to 2^32 / row_len, so a row sum reaches high bits and stays below 2^32; a tenth of them 0"""
    rng = np.random.default_rng([n_rows, row_len])
    m = n_rows * row_len
    data = np.full(m + 40, CANARY, np.uint32)
    data[:m] = rng.integers(0, ref.U32_MAX // max(row_len, 1) + 1, m, dtype=np.uint64) * (rng.random(m) >= 0.1)
    totals = np.full(n_rows + 3, CANARY, np.uint32)
    want, want_totals = ref.scan_rows(data, n_rows, row_len)
    (got, got_totals), launches = _launches(ctx, lambda: ctx.debug_scan_rows(data, n_rows, row_len, totals=totals))
    _same(got[:m], want, "scanned rows")
    _same(got[m:], data[m:], "words past the last row")
    _same(got_totals[:n_rows], want_totals, "row totals")
    _same(got_totals[n_rows:], totals[n_rows:], "words past the last total")
    assert launches == 1


# ---- run_heads -------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("pattern", ["equal", "distinct", "edge_256", "runs"])
@pytest.mark.parametrize("n", [1, 255, 256, 257, 3 * 2 ** 20 + 11])
def test_run_heads(ctx, n, pattern):
    rng = np.random.default_rng([n, len(pattern)])
    if pattern == "equal":
        s = np.full(n, 77, np.uint32)
    elif pattern == "distinct":
        s = np.arange(n, dtype=np.uint32) * np.uint32(3)
    elif pattern == "edge_256":  # one run boundary, exactly at the first block edge
        s = (np.arange(n) >= 256).astype(np.uint32)
    else:
        s = np.cumsum(rng.random(n) < 0.2).astype(np.uint32)
    canary = np.full(n + 8, CANARY, np.uint32)
    got, launches = _launches(ctx, lambda: ctx.debug_run_heads(s, head=canary))
    _same(got[:n], ref.run_heads(s), "head")
    _same(got[n:], canary[n:], "words past head[n - 1]")
    assert launches == 1


def test_run_heads_of_nothing(ctx):
    canary = np.full(8, CANARY, np.uint32)
    got, launches = _launches(ctx, lambda: ctx.debug_run_heads(np.zeros(0, np.uint32), head=canary))
    _same(got, canary, "head of an empty list")
    assert launches == 0
