"""The exact references of the sorted-key primitives (tests/sort_scan_reference.py) against brute-force loops, and the
argument checks of their parity hooks.  CPU only: these pin the yardstick tests/test_gpu_sort_scan.py holds the device to."""
import ctypes as C

import numpy as np
import pytest

import sort_scan_reference as ref


def _c_passes(max_key):
    """radix_sort_u32's own loop: bits = 1, grown while max_key >> bits is non-zero, at most 32; one pass per 8 bits"""
    bits = 1
    while bits < 32 and (max_key >> bits) != 0:
        bits += 1
    return (bits + 7) // 8


def test_pass_count_at_the_byte_boundaries():
    table = {0: 1, 1: 1, 255: 1, 256: 2, 2 ** 16 - 1: 2, 2 ** 16: 3, 2 ** 24 - 1: 3, 2 ** 24: 4, 2 ** 32 - 1: 4, 2 ** 32: 4,
             2 ** 40: 4, 2 ** 64 - 1: 4}
    for m, passes in table.items():
        assert ref.radix_passes(m) == passes == _c_passes(m), m
    for b in range(1, 64):
        for m in (2 ** b - 1, 2 ** b, 2 ** b + 1):
            assert ref.radix_passes(m) == _c_passes(m), m


def _insertion_sort(keys, payloads):
    """stable by construction: an element moves left only past strictly greater keys"""
    k, p = list(keys), [list(v) for v in payloads]
    for i in range(1, len(k)):
        j = i
        while j > 0 and k[j - 1] > k[j]:
            k[j - 1], k[j] = k[j], k[j - 1]
            for v in p:
                v[j - 1], v[j] = v[j], v[j - 1]
            j -= 1
    return k, p


@pytest.mark.parametrize("max_key", [0, 3, 255, 256, 2 ** 32 - 1, 2 ** 40])
def test_radix_sort_reference_is_a_stable_sort(max_key):
    rng = np.random.default_rng(max_key % 1000)
    for n in (0, 1, 2, 7, 40):
        hi = min(max_key, ref.U32_MAX)
        keys = rng.choice(np.array(sorted({0, hi // 2, hi}), np.uint32), n)
        v0, v1 = rng.integers(0, 2 ** 32, n, dtype=np.uint32), rng.integers(0, 2 ** 32, n, dtype=np.uint32)
        k, (p0, p1, idx) = _insertion_sort(keys.tolist(), [v0.tolist(), v1.tolist(), list(range(n))])
        rk, r0, r1, alt = ref.radix_sort(keys, max_key, v0, v1)
        assert rk.tolist() == k and r0.tolist() == p0 and r1.tolist() == p1
        assert alt == (n > 0 and _c_passes(max_key) % 2 == 1)
        rk, ri, rn, _ = ref.radix_sort(keys, max_key, v0, None, v0_iota=True)  # v0's contents are not used
        assert rk.tolist() == k and ri.tolist() == idx and rn is None


def test_lower_bounds_reference_against_a_linear_search():
    rng = np.random.default_rng(3)
    for n_keys, shift in ((0, 0), (5, 0), (9, 3), (16, 5), (256, 24), (2, 31), (3, 31)):
        top = min((n_keys + 1) << shift, 2 ** 32)  # keys reach past n_keys << shift, up to 2^32 - 1
        s = np.sort(rng.integers(0, top, 60, dtype=np.uint64)).astype(np.uint32)
        s[-1] = ref.U32_MAX
        for length in (None, 0, 17):
            lst = s[:length].tolist()
            want = [next((i for i, v in enumerate(lst) if v >= k << shift), len(lst)) for k in range(n_keys + 1)]
            assert ref.lower_bounds(s, n_keys, shift, length).tolist() == want, (n_keys, shift, length)
    # k << shift == 2^32: past every 32-bit key, so the offset is the length
    assert ref.lower_bounds(np.array([0, ref.U32_MAX], np.uint32), 256, 24)[256] == 2


def test_flag_scan_reference_counts_only_ones():
    rng = np.random.default_rng(5)
    for n in (0, 1, 2, 50):
        flags = rng.choice(np.array([0, 1, 1, 2, 3, ref.U32_MAX], np.uint32), n)
        rank, total = ref.flag_scan(flags)
        c, want = 0, []
        for f in flags.tolist():
            want.append(c)
            c += f == 1
        assert rank.tolist() == want and total == c


def test_scan_rows_and_run_heads_references():
    rng = np.random.default_rng(6)
    for n_rows, row_len in ((1, 0), (1, 1), (3, 5), (2, 9)):
        data = rng.integers(0, 2 ** 29, n_rows * row_len + 3, dtype=np.uint32)
        out, totals = ref.scan_rows(data, n_rows, row_len)
        for r in range(n_rows):
            c = 0
            for i in range(row_len):
                assert out[r * row_len + i] == c
                c += int(data[r * row_len + i])
            assert totals[r] == c
    for keys in ([], [4], [4, 4, 5, 5, 5, 9], list(range(6))):
        want = [1 if i == 0 or keys[i] != keys[i - 1] else 0 for i in range(len(keys))]
        assert ref.run_heads(np.array(keys, np.uint32)).tolist() == want


def _null_ctx_rejects(call, *args):
    """the hook with a NULL context: bad arguments fail before the context is looked at, so no device is touched"""
    from yolo_ppf_pose_estimation_b200 import capi
    rc = getattr(capi.lib(), call)(None, *args)
    assert rc == -1, (call, rc)  # B200PPF_ERR_INVALID
    assert "bad argument" in capi.lib().b200ppf_last_error(None).decode(), call


def _no_device_context():
    """a Context with no device behind it: its hooks pass a NULL context"""
    from yolo_ppf_pose_estimation_b200 import capi
    ctx = capi.Context.__new__(capi.Context)
    ctx._h = C.c_void_p()
    return ctx


def test_hooks_reject_bad_arguments_without_a_device():
    from yolo_ppf_pose_estimation_b200 import capi
    w = np.zeros(8, np.uint32)
    out = C.c_int(0)
    total = C.c_uint32(0)
    p = w.ctypes.data_as(C.c_void_p)
    # radix sort: NULL keys, half a payload pair, NULL result flag
    _null_ctx_rejects("b200ppf_debug_radix_sort", None, p, None, None, None, None, 8, 255, 0, C.byref(out))
    _null_ctx_rejects("b200ppf_debug_radix_sort", p, p, p, None, None, None, 8, 255, 0, C.byref(out))
    _null_ctx_rejects("b200ppf_debug_radix_sort", p, p, None, None, None, p, 8, 255, 0, C.byref(out))
    _null_ctx_rejects("b200ppf_debug_radix_sort", p, p, None, None, None, None, 8, 255, 0, None)
    # lower bounds: NULL list, NULL offsets, offsets cap below n_keys + 1, a device length past n, shift of 32
    _null_ctx_rejects("b200ppf_debug_lower_bounds", None, 8, -1, 3, 0, p, 8)
    _null_ctx_rejects("b200ppf_debug_lower_bounds", p, 8, -1, 3, 0, None, 8)
    _null_ctx_rejects("b200ppf_debug_lower_bounds", p, 8, -1, 8, 0, p, 8)
    _null_ctx_rejects("b200ppf_debug_lower_bounds", p, 8, 9, 3, 0, p, 8)
    _null_ctx_rejects("b200ppf_debug_lower_bounds", p, 8, -1, 3, 32, p, 8)
    # flag scan: NULL flags, NULL rank, rank cap below n, NULL total
    _null_ctx_rejects("b200ppf_debug_flag_scan", None, 8, p, 8, 0, C.byref(total))
    _null_ctx_rejects("b200ppf_debug_flag_scan", p, 8, None, 8, 0, C.byref(total))
    _null_ctx_rejects("b200ppf_debug_flag_scan", p, 8, p, 7, 1, C.byref(total))
    _null_ctx_rejects("b200ppf_debug_flag_scan", p, 8, p, 8, 0, None)
    # scan rows: NULL data, NULL totals, no rows, n_rows * row_len past the data cap (also past 32 bits), totals cap
    _null_ctx_rejects("b200ppf_debug_scan_rows", None, 2, 4, 8, p, 8)
    _null_ctx_rejects("b200ppf_debug_scan_rows", p, 2, 4, 8, None, 8)
    _null_ctx_rejects("b200ppf_debug_scan_rows", p, 0, 4, 8, p, 8)
    _null_ctx_rejects("b200ppf_debug_scan_rows", p, 3, 3, 8, p, 8)
    _null_ctx_rejects("b200ppf_debug_scan_rows", p, 2 ** 16, 2 ** 16, 8, p, 8)
    _null_ctx_rejects("b200ppf_debug_scan_rows", p, 2, 4, 8, p, 1)
    # run heads: NULL keys, NULL head, head cap below n
    _null_ctx_rejects("b200ppf_debug_run_heads", None, 8, p, 8)
    _null_ctx_rejects("b200ppf_debug_run_heads", p, 8, None, 8)
    _null_ctx_rejects("b200ppf_debug_run_heads", p, 8, p, 7)
    # the Context wrappers raise with the same message; outputs smaller than the range the primitive writes
    nc = _no_device_context()
    for call in (lambda: nc.debug_lower_bounds(w, 8, 0, offsets=np.zeros(8, np.uint32)),
                 lambda: nc.debug_flag_scan(w, rank=np.zeros(7, np.uint32)),
                 lambda: nc.debug_scan_rows(w, 3, 3),
                 lambda: nc.debug_scan_rows(w, 2, 4, totals=np.zeros(1, np.uint32)),
                 lambda: nc.debug_run_heads(w, head=np.zeros(7, np.uint32))):
        with pytest.raises(capi.B200PPFError, match="bad argument"):
            call()
    # good arguments reach the context check, which fails without a device
    for call in (lambda: nc.debug_radix_sort(w, 255, v0=w, v0_iota=True), lambda: nc.debug_lower_bounds(w, 7, 0),
                 lambda: nc.debug_flag_scan(w, host_total=True), lambda: nc.debug_scan_rows(w, 2, 4),
                 lambda: nc.debug_run_heads(w)):
        with pytest.raises(capi.B200PPFError, match="null context"):
            call()
