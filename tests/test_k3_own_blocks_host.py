"""The own cell's per-step rule (k3_vote.cu own_step) restated on the CPU against the per-entry rule it shortcuts
(ppf_math.cuh alpha_bin_phase, "the kernel's first look"): a step whose live entry words are all below sub_lo << 24 votes
every entry below the scene phase, one whose words are all above (sub_hi << 24) | 0xFFFFFF votes every entry above it,
and any other step decides per entry.  The step rule must never disagree with the per-entry rule, whatever the order
of the entries, and must apply exactly when every entry is settled on one side."""
import numpy as np

M32 = 0xFFFFFFFF
BELOW, ABOVE, FULL = 1, 2, 0


def per_entry(w, sub_lo, sub_hi):
    """alpha_bin_phase: rel = sub - sub_lo (unsigned); rel > span settles the entry, the sign of rel gives the side"""
    rel = ((w >> 24) - sub_lo) & M32
    span = sub_hi - sub_lo
    if rel > span:
        return ABOVE if (rel if rel < 1 << 31 else rel - (1 << 32)) > span else BELOW
    return FULL


def per_step(ws, sub_lo, sub_hi):
    """own_step: one unsigned compare per word against each limit; the warp takes a side when every word agrees"""
    below_lim, above_lim = (sub_lo << 24) & M32, ((sub_hi << 24) | 0xFFFFFF) & M32
    if all(w < below_lim for w in ws):
        return BELOW
    if all(w > above_lim for w in ws):
        return ABOVE
    return None


def sub_ranges():
    # the scene's own sub-phases span one or two values (the guard band is far below one sub-phase); both ends of the
    # cell included
    for lo in range(256):
        yield lo, lo
        if lo < 255:
            yield lo, lo + 1


def test_step_rule_matches_per_entry_rule_on_random_steps():
    rng = np.random.default_rng(3)
    for sub_lo, sub_hi in sub_ranges():
        for _ in range(40):
            n = int(rng.integers(1, 129))  # live lanes of one group of steps (a tail step has fewer)
            # words concentrated around the scene's own sub-phases, with the hot-word bits random
            subs = np.clip(sub_lo + rng.integers(-3, 4, n), 0, 255) if rng.random() < 0.5 else rng.integers(0, 256, n)
            ws = [int(s) << 24 | int(h) for s, h in zip(subs, rng.integers(0, 1 << 24, n))]
            sides = {per_entry(w, sub_lo, sub_hi) for w in ws}
            got = per_step(ws, sub_lo, sub_hi)
            if got is not None:
                assert sides == {got}, (sub_lo, sub_hi, got, sides)
            else:
                assert len(sides) > 1 or FULL in sides, (sub_lo, sub_hi, sides)


def test_step_rule_at_the_edges_of_the_own_sub_phases():
    for sub_lo, sub_hi in sub_ranges():
        edge_words = [0, 0xFFFFFF, M32, 0xFF000000]
        for s in (sub_lo - 1, sub_lo, sub_hi, sub_hi + 1):
            if 0 <= s <= 255:
                edge_words += [s << 24, s << 24 | 0xFFFFFF]
        for w in edge_words:
            side = per_entry(w, sub_lo, sub_hi)
            assert per_step([w], sub_lo, sub_hi) == (None if side == FULL else side), (hex(w), sub_lo, sub_hi)
        # sub_hi = 255: no word lies above; sub_lo = 0: none below
        if sub_hi == 255:
            assert per_step([M32], sub_lo, sub_hi) is None
        if sub_lo == 0:
            assert per_step([0], sub_lo, sub_hi) is None


def test_step_rule_does_not_depend_on_the_order():
    rng = np.random.default_rng(5)
    for sub_lo, sub_hi in [(0, 0), (0, 1), (31, 32), (32, 32), (127, 128), (254, 255), (255, 255)]:
        for _ in range(200):
            ws = [int(x) for x in rng.integers(0, 1 << 32, int(rng.integers(1, 129)), dtype=np.uint64)]
            got = per_step(ws, sub_lo, sub_hi)
            for _ in range(3):
                assert per_step(list(rng.permutation(ws)), sub_lo, sub_hi) == got
