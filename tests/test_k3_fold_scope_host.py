"""The flush model of tools/k3_fold_count.py on scenes small enough to follow by hand: where the kernel's sweep flushes the
candidate queue, which tasks fold, and which flushes one fold scope (one phase D) takes."""
import os
import sys

import numpy as np

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools"))
import k3_fold_count as fc  # noqa: E402


def one_cell_scene(n):
    """n points in one grid cell (radius 1): a corner at the bounding-box minimum, the rest inside [0.05, 0.5]^3"""
    rng = np.random.default_rng(7)
    P = np.zeros((n, 6), np.float32)
    P[1:, :3] = rng.uniform(0.05, 0.5, (n - 1, 3))
    return P


def test_flush_boundaries_one_cell():
    # 21 points, blocks of 4 in scene order, reference point 0 (not a candidate of itself); the 27 cells (21 points) overflow
    # a queue of 8, so the sweep flushes after a block once more than 8 - 4 candidates are buffered:
    #   block 0-3: 3 | 4-7: 7 -> flush | 8-11: 4 | 12-15: 8 -> flush | 16-19: 4 | 20: 5 -> flush | the final flush: empty
    scene = one_cell_scene(21)
    many, fl = fc.sweep_flushes(scene, 0, np.ones(21, bool), 1.0, threads=4, cand_cap=8)
    assert many
    assert fl == [list(range(1, 8)), list(range(8, 16)), list(range(16, 21)), []]
    # out-of-radius points are swept but not queued: without points 4-6 the first flush comes one block later
    #   0-3: 3 | 4-7: 4 | 8-11: 8 -> flush | 12-15: 4 | 16-19: 8 -> flush | 20: 1, the final flush
    inr = np.ones(21, bool)
    inr[[4, 5, 6]] = False
    many, fl = fc.sweep_flushes(scene, 0, inr, 1.0, threads=4, cand_cap=8)
    assert fl == [[1, 2, 3, 7, 8, 9, 10, 11], list(range(12, 20)), [20]]
    # a neighbourhood that fits the queue is one flush, whatever it holds
    many, fl = fc.sweep_flushes(scene[:8], 0, np.ones(8, bool), 1.0, threads=4, cand_cap=8)
    assert not many and fl == [list(range(1, 8))]


def test_far_cells_are_not_swept():
    scene = one_cell_scene(6)
    scene[5, :3] = (2.5, 0.2, 0.2)  # two cells away in x
    many, fl = fc.sweep_flushes(scene, 0, np.ones(6, bool), 1.0, threads=4, cand_cap=8)
    assert not many and fl == [[1, 2, 3, 4]]


def test_fold_gate_and_scopes():
    # single-flush tasks fold from FOLD_MIN_PAIRS candidates on
    assert fc.fold_scopes([fc.FOLD_MIN_PAIRS - 1], [900]) == []
    assert fc.fold_scopes([fc.FOLD_MIN_PAIRS], [900]) == [[0]]
    # a task that flushes more than once folds every flush, a short last one too; a scope ends once more than
    # FOLD_SCOPE - CAND_CAP = 6 144 codes are buffered: 1500 + 1400 + 1900 + 1700 = 6500
    assert fc.fold_scopes([1600, 1500, 2000, 1800, 300], [1500, 1400, 1900, 1700, 300]) == [[0, 1, 2, 3], [4]]
    # scopes end on codes, not candidates: pairs with an empty bucket leave none (1400 + 1300 + 1800 + 1600 = 6100)
    assert fc.fold_scopes([1600, 1500, 2000, 1800, 300], [1400, 1300, 1800, 1600, 300]) == [[0, 1, 2, 3, 4]]
    assert fc.fold_scopes([1300, 900], [1200, 800]) == [[0, 1]]
    # the hand-sized queue of the first test: scope 16, queue 8 -> a scope ends past 8 codes
    assert fc.fold_scopes([7, 8, 5, 0], [7, 8, 5, 0], fold_min=6, scope=16, cand_cap=8) == [[0, 1], [2, 3]]


def test_folded_words():
    # two pairs of one bucket (16 words, one per cell) with the same shift q, scene phases in cells 3 and 5: shift q is
    # voted on by cells 4..15 (12 words), shift q + 1 by cells 0..4 (5 words); one walk per pair is 2 x 15 words
    assert fc.fold_words([0, 0], [2, 2], [3, 5], [16, 16], 10) == 17
    code = {1: (0, 2, 3, 16.0), 2: (0, 2, 5, 16.0), 3: (1, 4, 0, 32.0)}
    w = fc.walked([[1, 2], [3]], code, 10)
    own = 64 / 16
    assert w["per_pair"] == 64
    # folding one flush at a time walks the two flushes apart; the scope and the task fold all three pairs together
    assert w["flush"] == own + 2 * 15 + 32 * 15 / 16  # both flushes are below FOLD_MIN_PAIRS: one walk per pair
    assert w["scope"] == w["task"] == own + 17 + 32 * 15 / 16
