"""Folded shift ranges (k3_vote.cu phase D), restated in NumPy: the groups the kernel forms from the sorted fold codes
(key, q, cell) and the multiplier m_s(k) it reads off them with lower bounds must cast, per (key, shift, cell), exactly
the votes that the per-pair walks cast — a pair (q, c) walks the cells below c with shift q + 1 (mod N_T) and the cells
above c with shift q."""
import numpy as np
import pytest


def per_pair(codes, qbits, lf, n_turn):
    """(key, s, k) -> number of pairs whose walk visits cell k of bucket key with shift s."""
    out = {}
    ncell = 1 << lf
    for code in codes.tolist():
        c, q, key = code & (ncell - 1), (code >> lf) & ((1 << qbits) - 1), code >> (lf + qbits)
        for k in range(ncell):
            if k == c:
                continue  # the pair's own cell: per-entry path
            s = q if k > c else (q + 1) % n_turn
            out[(key, s, k)] = out.get((key, s, k), 0) + 1
    return out


def folded(codes, qbits, lf, n_turn):
    """The kernel's phase D: sort, one group per (key, s) some run touches, m_s(k) from lower bounds."""
    ncell, qmask = 1 << lf, (1 << qbits) - 1
    srt = np.sort(np.asarray(codes, np.uint64))
    n = len(srt)
    lb = lambda x: int(np.searchsorted(srt, x, side="left"))  # noqa: E731
    groups = []
    for i in range(n):
        run = int(srt[i]) >> lf
        if i == 0 or (int(srt[i - 1]) >> lf) != run:
            q = run & qmask
            nxt = ((run - q) | (0 if q + 1 == n_turn else q + 1)) << lf
            p = lb(nxt)
            groups.append(run << lf)
            if p == n or (int(srt[p]) >> lf) != (nxt >> lf):
                groups.append(nxt)
    assert len(groups) == len(set(groups)), "a (key, s) group was formed twice"
    out = {}
    for g in groups:
        run = g >> lf
        s = run & qmask
        gp = ((run - s) | (n_turn - 1 if s == 0 else s - 1)) << lf
        A = [lb(g + k) for k in range(ncell)]
        B = [lb(gp + k) for k in range(1, ncell + 1)]
        for k in range(ncell):
            m = (A[k] - A[0]) + (B[ncell - 1] - B[k])
            if m:
                out[(run >> qbits, s, k)] = m
    return out


@pytest.mark.parametrize("n_turn,lf,seed", [(30, 4, 0), (30, 4, 1), (30, 3, 2), (2, 4, 3), (360, 2, 4), (31, 4, 5)])
def test_fold_multipliers_match_per_pair_walks(n_turn, lf, seed):
    rng = np.random.default_rng(seed)
    qbits = max(1, int(n_turn - 1).bit_length())
    for trial in range(20):
        n = int(rng.integers(1, 600))
        n_keys = int(rng.integers(1, 6))
        keys = rng.integers(0, 1 << 12, n_keys)[rng.integers(0, n_keys, n)]
        # q concentrated on few values (dense buckets) including the last position N_T - 1, whose walks below its
        # cell wrap to shift 0
        qs = rng.choice([0, n_turn - 1, int(rng.integers(0, n_turn)), int(rng.integers(0, n_turn))], n)
        cs = rng.integers(0, 1 << lf, n)
        codes = (((keys.astype(np.int64) << qbits) | qs) << lf) | cs
        assert int(codes.max()) < 1 << 31
        assert folded(codes, qbits, lf, n_turn) == per_pair(codes, qbits, lf, n_turn)


def test_fold_wraps_last_position_to_shift_zero():
    # one pair at q = N_T - 1 in cell 5 and one at q = 0 in cell 9: cells below 5 take shift 0 from the first pair,
    # cells above 9 take shift 0 from the second — one group (key, 0) with both
    n_turn, lf, qbits = 30, 4, 5
    codes = np.array([(((7 << qbits) | (n_turn - 1)) << lf) | 5, (((7 << qbits) | 0) << lf) | 9])
    f = folded(codes, qbits, lf, n_turn)
    assert f == per_pair(codes, qbits, lf, n_turn)
    assert all(f[(7, 0, k)] == 1 for k in list(range(5)) + list(range(10, 16)))
    # cells 6..8 lie above the first pair's cell (shift N_T - 1) and below the second's (shift 1)
    assert all((7, 0, k) not in f and f[(7, n_turn - 1, k)] == 1 and f[(7, 1, k)] == 1 for k in range(6, 9))
