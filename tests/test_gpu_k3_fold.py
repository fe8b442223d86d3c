"""Folded shift ranges (k3_vote.cu phase D): the constant-shift walks of the scene pairs of one reference point that share a
bucket and a shift are cast by one walk whose counts are multiplied by the number of such pairs.  These scenes put
hundreds of pairs into the same (key, q) of a table large enough to fold (2 009-point model, 4 M entries), and check the
full accumulators and the peaks bit-exact against the oracle's bucket walk on the device's own pair quantities."""
import numpy as np
import pytest

from conftest import ANGLE_STEP, DIST_STEP

pytestmark = pytest.mark.gpu

PLANE_Z = np.float32(0.55)  # just below the bottle (z 0.559 ... 0.681)


@pytest.fixture(scope="module")
def big_table(ctx, oracle, bottle_5mm):
    feats = oracle.ppf_estimation(bottle_5mm)
    hm = oracle.HashMap(ANGLE_STEP, DIST_STEP).set_input_feature_cloud(feats)
    t = ctx.table_build(ctx.features_upload(feats), ANGLE_STEP, DIST_STEP)
    assert t.info.n_entries == hm.num_entries >= 1 << 21 and t.info.phase_cells == 16
    return t, hm


def plane_patch(spacing=0.0025, lo=(-0.3, -0.3), hi=(0.2, 0.2)):
    xs = np.arange(lo[0], hi[0], spacing, dtype=np.float64)
    ys = np.arange(lo[1], hi[1], spacing, dtype=np.float64)
    X, Y = np.meshgrid(xs, ys, indexing="ij")
    P = np.zeros((X.size, 6), np.float32)
    P[:, 0], P[:, 1], P[:, 2], P[:, 5] = X.ravel(), Y.ravel(), PLANE_Z, 1.0
    return P


def check_refs(ctx, t, hm, n_model, ds, refs, min_pairs=0):
    for s_r in refs:
        inr, d, a = ctx.vote_debug_pairs(t, ds, int(s_r))
        assert inr.sum() >= min_pairs, (s_r, int(inr.sum()))
        acc = ctx.vote_debug_accumulator(t, ds, int(s_r))
        ref, votes = hm.vote_accumulate_from_pairs(n_model, d[inr > 0], a[inr > 0])
        assert votes == int(acc.sum()), (s_r, votes, int(acc.sum()))
        assert np.array_equal(acc, ref), f"accumulator differs for reference {s_r}"
        # the votes counter still adds the whole bucket of every pair
        assert ctx.vote_stats()["votes"] == votes


def check_peaks(ctx, t, dm, ds, first, step, count):
    hy = ctx.vote(dm, t, ds, first, step, count)
    for h in hy:
        acc = ctx.vote_debug_accumulator(t, ds, int(h["scene_index"]))
        flat = int(np.argmax(acc))
        assert h["votes"] == acc.reshape(-1)[flat]
        if h["votes"]:
            assert (int(h["model_index"]), int(h["alpha_bin"])) == divmod(flat, acc.shape[1])


def test_fold_plane_and_object(ctx, bottle_5mm, big_table):
    """A dense planar patch (2.5 mm grid: ~4 300 in-radius neighbours per plane point, so the candidate queue flushes
    several times and each flush folds on its own) with the bottle standing on it."""
    t, hm = big_table
    plane = plane_patch()
    scene = np.concatenate([plane, bottle_5mm]).astype(np.float32)
    ds = ctx.upload_cloud(scene)
    n_plane = plane.shape[0]
    # plane points under / beside the object and far from it, object points
    near = int(np.argmin(np.linalg.norm(plane[:, :2] - np.array([-0.06, -0.05], np.float32), axis=1)))
    far = int(np.argmin(np.linalg.norm(plane[:, :2] - np.array([-0.2, 0.1], np.float32), axis=1)))
    refs = [near, far, n_plane + 0, n_plane + 1000, n_plane + 2008]
    check_refs(ctx, t, hm, bottle_5mm.shape[0], ds, refs[:2], min_pairs=3000)
    check_refs(ctx, t, hm, bottle_5mm.shape[0], ds, refs[2:])
    dm = ctx.upload_cloud(bottle_5mm)
    check_peaks(ctx, t, dm, ds, near, 1, 3)
    check_peaks(ctx, t, dm, ds, n_plane + 500, 401, 4)


def _rotate_z(P, centre, theta):
    c, s = np.cos(theta), np.sin(theta)
    R = np.array([[c, -s, 0.0], [s, c, 0.0], [0.0, 0.0, 1.0]])
    out = np.empty_like(P)
    out[:, :3] = ((P[:, :3].astype(np.float64) - centre) @ R.T + centre).astype(np.float32)
    out[:, 3:] = (P[:, 3:].astype(np.float64) @ R.T).astype(np.float32)
    return out


def test_fold_scene_phases_at_cell_and_bin_edges(ctx, bottle_5mm, big_table):
    """Object points copied around the reference point's normal: the pair features (so the bucket) stay, the scene
    phase moves.  The copies put scene phases within a few 1e-7 rad of phase-cell and bin edges — pairs that fall back
    to the per-entry walk — next to pairs inside their cells and duplicates of them, which fold, all in one bucket."""
    t, hm = big_table
    plane = plane_patch()
    n_plane = plane.shape[0]
    s_r = int(np.argmin(np.linalg.norm(plane[:, :2] - np.array([-0.06, -0.05], np.float32), axis=1)))
    centre = plane[s_r, :3].astype(np.float64)
    # object points within the radius of the reference point
    radius = 0.5 * float(t.info.max_dist)
    dist = np.linalg.norm(bottle_5mm[:, :3] - plane[s_r, :3], axis=1)
    base = bottle_5mm[np.flatnonzero(dist < 0.8 * radius)[::97][:10]]
    assert len(base) >= 5
    # the scene phase of each base point, and which way a rotation about the normal moves it
    probe = np.concatenate([plane, base, _rotate_z(base, centre, 0.01)]).astype(np.float32)
    inr, _, a = ctx.vote_debug_pairs(t, ctx.upload_cloud(probe), s_r)
    a0 = a[n_plane:n_plane + len(base)].astype(np.float64)
    a1 = a[n_plane + len(base):].astype(np.float64)
    assert inr[n_plane:].all()
    sign = np.sign(np.median(a1 - a0))
    step = float(ANGLE_STEP)
    copies = []
    for b, alpha in zip(base, a0):
        u = alpha / step
        edges = [(np.floor(u * 16) + j) / 16 for j in range(-3, 4)] + [np.round(u) - 1, np.round(u) + 1]
        for e in edges:
            for eps in (-3e-6, -4e-7, 0.0, 4e-7, 3e-6, step / 40):
                theta = sign * (e * step + eps - alpha)
                c = _rotate_z(b[None], centre, theta)
                copies += [c, c] if eps == step / 40 else [c]  # duplicates: identical pairs fold with multiplicity
    scene = np.concatenate([plane] + copies).astype(np.float32)
    ds = ctx.upload_cloud(scene)
    inr, d, a = ctx.vote_debug_pairs(t, ds, s_r)
    ac = a[n_plane:].astype(np.float64)
    ph = (ac / step) * 16
    near_edge = np.abs(ph - np.round(ph)) * step / 16 < 4e-6
    assert near_edge.sum() > 50 and (~near_edge).sum() > 50
    check_refs(ctx, t, hm, bottle_5mm.shape[0], ds, [s_r], min_pairs=2048)
    check_peaks(ctx, t, ctx.upload_cloud(bottle_5mm), ds, s_r, 1, 1)
