"""Exact references of the sorted-key primitives (csrc/sort_scan.cu): plain NumPy on int64 / uint64, where no sum, shift or
target can wrap.  tests/test_gpu_sort_scan.py holds the device to these bit for bit; tests/test_sort_scan_reference_host.py
checks them against brute-force loops.

Every function takes host arrays of uint32 words, as the parity hooks do, and returns what the primitive documents:
  radix_sort     stable ascending order of the keys (argsort kind="stable" fixes the payload order exactly); the result
                 is in the alternate buffers when the pass count is odd
  lower_bounds   offsets[k] = first i with sorted[i] >= k << shift, k = 0 .. n_keys
  flag_scan      rank[k] = flags equal to 1 before k, and their total
  scan_rows      exclusive scan of each row, and its sum
  run_heads      1 where a run of equal keys starts
"""
import numpy as np

U32_MAX = 2 ** 32 - 1


def radix_passes(max_key):
    """8-bit passes of a sort whose largest key is max_key: one per byte of its bits (max_key clamped to 32 bits), at
    least one"""
    bits = min(int(max_key), U32_MAX).bit_length()
    return max(1, -(-bits // 8))


def radix_sort(keys, max_key, v0=None, v1=None, v0_iota=False):
    """-> (keys, v0, v1, result_in_alt): keys ascending, stable, payloads carried along (None when not given); v0_iota
    takes v0 to be 0..n-1.  Every key must be <= max_key: the sort orders max_key's bits only."""
    k = np.asarray(keys, np.uint32).astype(np.int64)
    assert k.size == 0 or int(k.max()) <= int(max_key), "a key above max_key"
    order = np.argsort(k, kind="stable")
    if v0 is not None and v0_iota:
        v0 = np.arange(k.size, dtype=np.uint32)
    v0, v1 = (None if v is None else np.asarray(v, np.uint32)[order] for v in (v0, v1))
    in_alt = k.size > 0 and radix_passes(max_key) % 2 == 1
    return k[order].astype(np.uint32), v0, v1, in_alt


def lower_bounds(sorted_keys, n_keys, shift, length=None):
    """offsets (n_keys + 1 words) into sorted_keys[:length] (all of it for None); targets k << shift as exact int64
    (n_keys < 2^32 and shift < 32 keep them below 2^63)"""
    s = np.asarray(sorted_keys, np.uint32)[:length].astype(np.int64)
    assert np.all(s[1:] >= s[:-1]), "the list must be sorted"
    assert 0 <= n_keys <= U32_MAX and 0 <= shift < 32
    targets = np.arange(n_keys + 1, dtype=np.int64) << shift
    return np.searchsorted(s, targets, side="left").astype(np.uint32)


def flag_scan(flags):
    """-> (rank, total): only flags equal to 1 count"""
    ones = (np.asarray(flags, np.uint32) == 1).astype(np.int64)
    incl = np.cumsum(ones)
    return (incl - ones).astype(np.uint32), int(incl[-1]) if ones.size else 0


def scan_rows(data, n_rows, row_len):
    """-> (scanned rows, n_rows * row_len words; totals, n_rows words) of the first n_rows * row_len words of data.  A row
    sum must stay below 2^32: the primitive's words are 32-bit"""
    d = np.asarray(data, np.uint32)[:n_rows * row_len].astype(np.uint64).reshape(n_rows, row_len)
    incl = np.cumsum(d, axis=1, dtype=np.uint64)
    totals = incl[:, -1] if row_len else np.zeros(n_rows, np.uint64)
    assert np.all(totals <= U32_MAX), "a row sum past 32 bits"
    return (incl - d).astype(np.uint32).reshape(-1), totals.astype(np.uint32)


def run_heads(sorted_keys):
    s = np.asarray(sorted_keys, np.uint32).astype(np.int64)
    head = np.ones(s.size, np.uint32)
    head[1:] = np.diff(s) != 0
    return head
