"""Fold scopes (k3_vote.cu phase D): a task's fold codes collect across the flushes of its candidate queue and are folded
once FOLD_SCOPE - CAND_CAP are buffered after a flush, and at the end of the task; a task that flushes more than once folds
every flush, a short last one too.  Full accumulators and peaks bit-exact against the oracle's bucket walk on the device's
own pair quantities, on the 4 M-entry table of the 2 009-point model and planar patches under it."""
import os
import sys

import numpy as np
import pytest

from test_gpu_k3_fold import big_table, check_peaks, check_refs, plane_patch  # noqa: F401  (big_table: fixture)

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools"))
import k3_fold_count as fc  # noqa: E402

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def buckets(big_table):
    _, hm = big_table
    keys, _ = hm.dump_keys()
    return {tuple(k) for k in keys.tolist()}


def nonempty_pairs(ctx, t, ds, s_r, buckets):
    inr, d, _ = ctx.vote_debug_pairs(t, ds, s_r)
    return inr, sum(1 for x in d[inr > 0].tolist() if tuple(x) in buckets)


def test_fold_scope_ends_mid_task(ctx, bottle_5mm, big_table, buckets):
    """A 1.5 mm plane under the bottle: more than FOLD_SCOPE pairs with a non-empty bucket around one reference point, so
    phase D runs before the task ends and again at its end."""
    t, hm = big_table
    plane = plane_patch(spacing=0.0015)
    scene = np.concatenate([plane, bottle_5mm]).astype(np.float32)
    ds = ctx.upload_cloud(scene)
    s_r = int(np.argmin(np.linalg.norm(plane[:, :2] - np.array([-0.06, -0.05], np.float32), axis=1)))
    inr, n = nonempty_pairs(ctx, t, ds, s_r, buckets)
    assert n > fc.FOLD_SCOPE, n  # more codes than one scope holds
    check_refs(ctx, t, hm, bottle_5mm.shape[0], ds, [s_r], min_pairs=fc.FOLD_SCOPE)
    check_peaks(ctx, t, ctx.upload_cloud(bottle_5mm), ds, s_r, 1, 2)


def test_short_last_flush_folds(ctx, bottle_5mm, big_table):
    """Plane points whose task flushes more than once and whose last flush holds fewer than FOLD_MIN_PAIRS candidates (by
    the sweep's flush model): that flush folds with the others."""
    t, hm = big_table
    plane = plane_patch()
    scene = np.concatenate([plane, bottle_5mm]).astype(np.float32)
    ds = ctx.upload_cloud(scene)
    radius = 0.5 * float(t.info.max_dist)
    found = []
    for s_r in range(0, plane.shape[0], 997):
        inr, _, _ = ctx.vote_debug_pairs(t, ds, s_r)
        _, flushes = fc.sweep_flushes(scene, s_r, inr > 0, radius)
        if len(flushes) > 1 and 0 < len(flushes[-1]) < fc.FOLD_MIN_PAIRS:
            found.append(s_r)
        if len(found) == 3:
            break
    assert found
    check_refs(ctx, t, hm, bottle_5mm.shape[0], ds, found, min_pairs=fc.CAND_CAP - fc.THREADS)


def test_vote_many_references(ctx, bottle_5mm, big_table):
    """One vote over many reference points of plane and object: persistent CTAs run several tasks each, light and folding
    ones, each in its CTA's slot of the fold buffer."""
    t, _ = big_table
    plane = plane_patch()
    scene = np.concatenate([plane, bottle_5mm]).astype(np.float32)
    ds = ctx.upload_cloud(scene)
    check_peaks(ctx, t, ctx.upload_cloud(bottle_5mm), ds, 5, 211, scene.shape[0] // 211)
