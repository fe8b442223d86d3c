"""K6 (k6_icp.cu) step by step: the device ICP after each of its first iterations, against the float64 NumPy restatement
(tests/icp_reference.py) and the CPU oracle, on every nearest-neighbour search path, grid-sizing branch and cluster size.

tolerance = 0 switches the stop test off, so max_iterations and num_levels fix how many iterations run on which level.
Every case first checks that no decision of the restatement (nearest neighbour, rejection, winner, solve branch) sits on
a tie that a last-bit difference could flip; then the device must run exactly as many iterations and end within 1e-9
of the restatement (rotation entries; translation relative to the scene's extent; residual relative).  What may differ
is only the order of the double reductions and libm's sin / cos: about 1e-13.
"""
import numpy as np
import pytest

import icp_reference as ir

pytestmark = pytest.mark.gpu

TOL = 1e-9


def _rot(axis, ang):
    axis = np.asarray(axis, np.float64) / np.linalg.norm(axis)
    K = np.array([[0, -axis[2], axis[1]], [axis[2], 0, -axis[0]], [-axis[1], axis[0], 0]])
    return np.eye(3) + np.sin(ang) * K + (1 - np.cos(ang)) * K @ K


def _pose(axis=(0.3, 1.0, 0.2), ang=0.0, t=(0.0, 0.0, 0.0), about=None):
    """rotation by ang about axis through the point about, then translation t"""
    P = np.eye(4)
    P[:3, :3] = _rot(axis, ang) if ang else np.eye(3)
    c = np.zeros(3) if about is None else np.asarray(about, np.float64)
    P[:3, 3] = c - P[:3, :3] @ c + np.asarray(t, np.float64)
    return P


def _unit(v):
    return v / np.linalg.norm(v, axis=1, keepdims=True)


def grid_cell(scene_samples):
    """the cell edge the kernel picks for a level's scene samples (float32, as the kernel sizes it)"""
    s = scene_samples[:, :3].astype(np.float32)
    ex, ey, ez = (max(np.float32(s[:, c].max() - s[:, c].min()), np.float32(1e-9)) for c in range(3))
    md = np.float32(s.shape[0])
    cell = np.cbrt(ex * ey * ez / max(np.float32(1), min(np.float32(0.5) * md, np.float32(8192))))
    cell = max(np.float32(cell), max(ex, ey, ez) / np.float32(256))
    grows = 0
    while True:
        dims = [int(np.floor(e / cell)) + 1 for e in (ex, ey, ez)]
        if dims[0] * dims[1] * dims[2] <= 1 << 16:
            return cell, dims, grows
        cell = np.float32(cell * np.float32(1.26))
        grows += 1


# ---- clouds (fixed seeds) ---------------------------------------------------------------------------------------------
_CACHE = {}


def _synth(n_model, n_scene_pts=20000, radius=0.2):
    """a synthetic bottle of n_model points and the neighbourhood of its instance in the synthetic scene"""
    key = ("synth", n_model, n_scene_pts, radius)
    if key not in _CACHE:
        from yolo_ppf_pose_estimation_b200 import synth
        model = synth.synth_model(n_model, 1)
        G = synth.gt_pose(2)
        sc = synth.synth_scene(n_scene_pts, 2, model_seed=1)
        centre = G[:3, 3] + G[:3, :3] @ np.array([0.0, 0.0, 0.09])
        scene = sc[np.linalg.norm(sc[:, :3] - centre, axis=1) < radius]
        _CACHE[key] = (model, scene, G, centre)
    return _CACHE[key]


def _near_start(G, centre, k=0):
    return _pose((0.3, 1.0, 0.2 + 0.3 * k), 0.08, (0.008, -0.006, 0.004), about=centre) @ G


def case_synth(n_model=1500, n_scene=None, k=0):
    """synthetic bottle against the scene around its instance; n_scene keeps the first n_scene scene points"""
    model, scene, G, centre = _synth(n_model, 60000 if (n_scene or 0) > 3000 else 20000,
                                     0.25 if (n_scene or 0) > 3000 else 0.2)
    if n_scene is not None:
        assert scene.shape[0] >= n_scene, scene.shape
        scene = scene[:n_scene]
    return model, scene, _near_start(G, centre, k)


def case_far(cells=20.0):
    """the start pose moves the model ~cells grid cells off the scene: every query lies outside the grid"""
    model, scene, G, centre = _synth(1500)
    cell, _, _ = grid_cell(scene)
    lo, hi = scene[:, :3].min(axis=0), scene[:, :3].max(axis=0)
    shift = np.array([hi[0] - lo[0], 0.0, 0.0]) + cells * float(cell)
    return model, scene, _pose(t=shift) @ _near_start(G, centre), cells


def case_flat():
    """a square patch of a plane z = 0.9 (z extent 0: the 1e-9 clamp; 257 x 257 x 1 cells exceed ICP_CELLS_MAX) and a
    smaller patch of the same plane as the model"""
    from yolo_ppf_pose_estimation_b200 import synth
    u = synth.uniform(31, 0, 3000)
    v = synth.uniform(31, 1, 3000)
    xy = np.stack([0.3 * u, 0.3 * v], axis=1)
    xy[:4] = [[0, 0], [0.3, 0], [0, 0.3], [0.3, 0.3]]  # equal x and y extents
    scene = np.zeros((3000, 6), np.float32)
    scene[:, :2], scene[:, 2], scene[:, 5] = xy, 0.9, 1.0
    mu = synth.uniform(32, 0, 800)
    mv = synth.uniform(32, 1, 800)
    model = np.zeros((800, 6), np.float32)
    model[:, 0], model[:, 1], model[:, 2], model[:, 5] = 0.1 + 0.1 * mu, 0.1 + 0.1 * mv, 0.9, 1.0
    return model, scene, _pose((0.2, 0.1, 1.0), 0.05, (0.004, -0.003, 0.002), about=(0.15, 0.15, 0.9))


def case_needle():
    """a rod 0.6 m long and 2 mm thick (x extent 300 times y and z): its cells are sized by the 256-per-axis floor"""
    from yolo_ppf_pose_estimation_b200 import synth
    n = 2400
    scene = np.zeros((n, 6), np.float64)
    scene[:, 0] = 0.6 * synth.uniform(41, 0, n)
    scene[:, 1] = 0.002 * synth.uniform(41, 1, n)
    scene[:, 2] = 0.002 * synth.uniform(41, 2, n)
    scene[:2, :3] = [[0, 0, 0], [0.6, 0.002, 0.002]]
    scene[:, 3:] = _unit(np.stack([synth.normal(41, 3 + 2 * c, n) for c in range(3)], axis=1))
    scene = scene.astype(np.float32)
    model = scene[(scene[:, 0] > 0.2) & (scene[:, 0] < 0.3)][::2]
    return model, scene, _pose((1.0, 0.2, 0.1), 0.002, (0.0004, 0.0002, -0.0002), about=(0.25, 0.001, 0.001))


def case_duplicate_scene():
    """every scene point twice (the copy about 8 places after the original): nearest-neighbour ties go to the lower index"""
    model, scene, start = case_synth(1500)
    dup = np.concatenate([scene, scene])
    order = np.argsort(np.concatenate([np.arange(len(scene)) * 2, np.arange(len(scene)) * 2 + 15]), kind="stable")
    return model, dup[order], start


def case_small_scene():
    """a 300-point scene under a model with every point twice: winners tie exactly and go to the lower model sample"""
    model, scene, start = case_synth(1500)
    m2 = np.repeat(model[:750], 2, axis=0)
    return m2, scene[::7][:300], start


def case_half_zero():
    """the scene holds 749 of the 1 500 model samples exactly: at the identity start their squared distances are 0"""
    model, scene, _ = case_synth(1500)
    rng = np.random.default_rng(5)
    moved = model.copy()
    moved[749:, :3] += rng.normal(scale=0.002, size=(751, 3)).astype(np.float32)
    sc = np.concatenate([model[:749], scene])
    return moved, sc, np.eye(4)


def case_zero_normal():
    model, scene, start = case_synth(1500)
    scene = scene.copy()
    scene[::7, 3:] = 0.0
    return model, scene, start


def case_few_pairs():
    """a 6-point model: after the rejection four pairs survive (the minimum-norm branch)"""
    model, scene, start = case_synth(1500)
    return model[::250][:6], scene, start


# ---- the comparison ---------------------------------------------------------------------------------------------------

def _tight(ctx, oracle, name, model, scene, start, max_iterations, num_levels, rejection_scale=2.5, min_iterations=1):
    """device vs restatement vs oracle for one start pose, tolerance 0; returns (device pose, restatement result)"""
    ref = ir.register(model, scene, start, max_iterations, 0.0, rejection_scale, num_levels)
    margins = ref.margins()
    for k, v in margins.items():
        if k != "fperc_gap":  # with tolerance 0 the stop test cannot fire: its margin decides nothing
            assert v > 0, (name, k, v)
    assert ref.iterations >= min_iterations, (name, ref.iterations)
    R, rres, rit = oracle.icp_refine(model, scene, start[None], max_iterations, 0.0, rejection_scale, num_levels)
    P, res, it = ctx.icp_refine(ctx.upload_cloud(model), ctx.upload_cloud(scene), start[None], max_iterations, 0.0,
                                rejection_scale, num_levels)
    assert it == ref.iterations == rit, (name, it, ref.iterations, rit)
    ext = float((scene[:, :3].max(axis=0) - scene[:, :3].min(axis=0)).max())
    d_rot = float(np.abs(P[0, :3, :3] - ref.pose[:3, :3]).max())
    d_t = float(np.abs(P[0, :3, 3] - ref.pose[:3, 3]).max()) / ext
    d_res = abs(res[0] - ref.residual) / max(abs(ref.residual), 1e-300)
    o_rot = float(np.abs(R[0, :3, :3] - ref.pose[:3, :3]).max())
    o_t = float(np.abs(R[0, :3, 3] - ref.pose[:3, 3]).max()) / ext
    print(f"ICP-STEPS {name}: iterations {it} branches {sorted(set(t.branch for t in ref.trace))} "
          f"device-ref rot {d_rot:.3g} t/extent {d_t:.3g} residual {d_res:.3g} | oracle-ref rot {o_rot:.3g} t {o_t:.3g} | "
          + " ".join(f"{k} {v:.3g}" for k, v in margins.items()))
    assert d_rot <= TOL and d_t <= TOL and d_res <= TOL, (name, d_rot, d_t, d_res)
    assert o_rot <= TOL and o_t <= TOL and abs(rres[0] - ref.residual) <= TOL * max(abs(ref.residual), 1e-300)
    return P[0], ref


# ---- search paths -----------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("max_iterations", [1, 2, 3, 6])
@pytest.mark.parametrize("n_scene", [1024, 1025])
def test_brute_force_and_grid_at_one_level(ctx, oracle, n_scene, max_iterations):
    """1 024 scene samples are searched from shared memory, 1 025 through the grid (unseeded first, then seeded by the
    previous iteration's match)"""
    model, scene, start = case_synth(1500, n_scene)
    _tight(ctx, oracle, f"one level, {n_scene} scene samples, {max_iterations} it", model, scene, start,
           max_iterations, 1)


@pytest.mark.parametrize("max_iterations", [1, 2, 3])
def test_grid_at_every_level(ctx, oracle, max_iterations):
    """3 levels, 4 400 scene points: the coarsest level (1 100 samples) searches the grid unseeded, the finer ones seeded
    from the coarser level's matches; max_iterations 3 runs 1 + 2 + 3 iterations"""
    model, scene, start = case_synth(2000, 4400)
    ref = ir.register(model, scene, start, max_iterations, 0.0, 2.5, 3)
    assert min(md for _, _, md, _, _ in ref.levels) > 1024, ref.levels
    _tight(ctx, oracle, f"three grid levels, {max_iterations} it", model, scene, start, max_iterations, 3)


@pytest.mark.parametrize("cells", [10.0, 30.0])
def test_start_off_the_grid(ctx, oracle, cells):
    """the model starts 10 / 30 cells beyond the scene's bounding box: the cube search grows until it reaches it"""
    model, scene, start, _ = case_far(cells)
    assert ir.transform_cloud(model, start)[:, 0].min() > scene[:, 0].max()
    _tight(ctx, oracle, f"start {cells:.0f} cells off the grid", model, scene, start, 2, 1)


# ---- grid sizing ------------------------------------------------------------------------------------------------------

def test_flat_scene(ctx, oracle):
    """z extent 0 -> the 1e-9 clamp; the first grid (257 x 257 x 1) is too large, the 1.26 growth runs; the plane leaves
    three of the six unknowns free (minimum-norm branch)"""
    model, scene, start = case_flat()
    _, dims, grows = grid_cell(scene)
    assert grows >= 1 and dims[2] == 1, (dims, grows)
    _, ref = _tight(ctx, oracle, "flat scene", model, scene, start, 3, 1)
    assert {t.branch for t in ref.trace} == {"min_norm"}


def test_needle_scene(ctx, oracle):
    """one axis 300 times the others: the cell is max extent / 256"""
    model, scene, start = case_needle()
    s = scene[:, :3].astype(np.float32)
    cell, dims, grows = grid_cell(scene)
    assert cell == np.float32(s[:, 0].max() - s[:, 0].min()) / np.float32(256) and grows == 0, (cell, dims)
    _tight(ctx, oracle, "needle scene", model, scene, start, 3, 1)


# ---- cluster sizes ----------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("n_model", [1024, 1025, 2049, 4097, 9000])
def test_cluster_sizes(ctx, oracle, n_model):
    """one CTA per 1 024 model points: clusters of 1, 2, 4, 8 and 8 CTAs"""
    model, scene, start = case_synth(n_model, 1500)
    _tight(ctx, oracle, f"model {n_model}", model, scene, start, 3, 2)


def test_forced_cluster_sizes_agree(ctx, oracle, monkeypatch):
    """the same input on 1, 2, 4 and 8 CTAs: the reductions change order only"""
    model, scene, start = case_synth(2049, 1500)
    dm, ds = ctx.upload_cloud(model), ctx.upload_cloud(scene)
    out = {}
    for cs in (1, 2, 4, 8):
        monkeypatch.setenv("B200PPF_ICP_CLUSTER", str(cs))
        out[cs] = ctx.icp_refine(dm, ds, start[None], 3, 0.0, 2.5, 2)
    monkeypatch.delenv("B200PPF_ICP_CLUSTER")
    ref = ir.register(model, scene, start, 3, 0.0, 2.5, 2)
    worst = 0.0
    for cs, (P, res, it) in out.items():
        assert it == ref.iterations, (cs, it, ref.iterations)
        d = float(np.abs(P[0] - out[1][0][0]).max())
        worst = max(worst, d, abs(res[0] - out[1][1][0]) / out[1][1][0])
        assert d <= 1e-12 and abs(res[0] - out[1][1][0]) <= 1e-12 * out[1][1][0], (cs, d)
        assert float(np.abs(P[0] - ref.pose).max()) <= TOL
    print(f"ICP-STEPS forced cluster sizes: largest difference to 1 CTA {worst:.3g}")


# ---- ties, built exactly ----------------------------------------------------------------------------------------------

def test_duplicate_scene_points(ctx, oracle):
    model, scene, start = case_duplicate_scene()
    _tight(ctx, oracle, "duplicate scene points", model, scene, start, 3, 2)


def test_scene_smaller_than_model_with_tied_winners(ctx, oracle):
    model, scene, start = case_small_scene()
    _tight(ctx, oracle, "small scene, tied winners", model, scene, start, 3, 1)


@pytest.mark.parametrize("n_model", [1500, 1501])
def test_even_and_odd_sample_counts(ctx, oracle, n_model):
    """m even and odd: the lower median is sample (m - 1) / 2 of the order"""
    model, scene, start = case_synth(n_model, 1500)
    _tight(ctx, oracle, f"m = {n_model}", model, scene, start, 3, 1)


def test_half_the_distances_zero(ctx, oracle):
    """749 of 1 500 squared distances are exactly 0: the median lands on the first non-zero one, the selects walk the
    zeros' histogram bins"""
    model, scene, start = case_half_zero()
    ref = ir.register(model, scene, start, 1, 0.0, 2.5, 1)
    _, d2, _ = ir.nearest(ir.transform_cloud(model, start)[:, :3], scene)
    assert (d2 == 0).sum() >= 749
    _tight(ctx, oracle, "half the distances zero", model, scene, start, 3, 1)
    assert ref.iterations == 1


# ---- degenerate cases -------------------------------------------------------------------------------------------------

def test_exact_fit_runs_no_iteration(ctx, oracle):
    """scene = model at the identity: every d2 is 0, so is the threshold, d2 < 0 rejects every pair"""
    model, _, _ = case_synth(1500)
    start = np.eye(4)
    P, res, it = ctx.icp_refine(ctx.upload_cloud(model), ctx.upload_cloud(model), start[None], 6, 0.0, 2.5, 3)
    R, _, rit = oracle.icp_refine(model, model, start[None], 6, 0.0, 2.5, 3)
    ref = ir.register(model, model, start, 6, 0.0, 2.5, 3)
    assert it == rit == ref.iterations == 0
    assert np.array_equal(P[0], start) and np.array_equal(R[0], start) and np.array_equal(ref.pose, start)


def test_one_point_model_and_scene(ctx, oracle):
    """the median is the only d2: the pair is rejected, no iteration runs, the start comes back unchanged"""
    model = np.array([[0.1, 0.2, 0.9, 0.0, 0.0, 1.0]], np.float32)
    scene = np.array([[0.12, 0.19, 0.91, 0.0, 0.6, 0.8]], np.float32)
    start = _pose((0.1, 0.2, 1.0), 0.3, (0.01, 0.02, -0.03))
    P, res, it = ctx.icp_refine(ctx.upload_cloud(model), ctx.upload_cloud(scene), start[None], 3, 0.0, 2.5, 2)
    R, _, rit = oracle.icp_refine(model, scene, start[None], 3, 0.0, 2.5, 2)
    ref = ir.register(model, scene, start, 3, 0.0, 2.5, 2)
    assert it == rit == ref.iterations == 0
    assert np.array_equal(P[0], start) and np.array_equal(R[0], start) and np.array_equal(ref.pose, start)


def test_levels_without_samples(ctx, oracle):
    """16 levels on 1 500 points: levels 15-12 hold no sample and are skipped, 11-3 run no iteration"""
    model, scene, start = case_synth(1500, 1500)
    ref = ir.register(model, scene, start, 2, 0.0, 2.5, 16)
    assert max(lv for lv, _, _, _, _ in ref.levels) == 11
    _tight(ctx, oracle, "16 levels", model, scene, start, 2, 16)


def test_fewer_than_six_pairs(ctx, oracle):
    model, scene, start = case_few_pairs()
    _, ref = _tight(ctx, oracle, "fewer than six pairs", model, scene, start, 3, 1)
    assert all(t.matches < 6 and t.branch == "min_norm" for t in ref.trace), [(t.matches, t.branch) for t in ref.trace]


def test_no_rejection(ctx, oracle):
    model, scene, start = case_synth(1500, 1500)
    _, ref = _tight(ctx, oracle, "rejection_scale 0", model, scene, start, 3, 2, rejection_scale=0.0)
    assert all(t.threshold == np.inf for t in ref.trace)


def test_level_budget_rounds_half_to_even(ctx, oracle):
    """max_iterations 5 over 4 levels: round(5/4), round(5/3), round(5/2) = 2 (not 3), 5"""
    model, scene, start = case_synth(1500, 1500)
    ref = ir.register(model, scene, start, 5, 0.0, 2.5, 4)
    assert [mi for _, _, _, _, mi in ref.levels] == [1, 2, 2, 5]
    _tight(ctx, oracle, "5 iterations over 4 levels", model, scene, start, 5, 4)


def test_scene_samples_with_zero_normals(ctx, oracle):
    model, scene, start = case_zero_normal()
    _tight(ctx, oracle, "zero scene normals", model, scene, start, 3, 2)


# ---- invariance, bitwise ----------------------------------------------------------------------------------------------

def test_batch_and_repeat_are_bitwise_invariant(ctx):
    """a pose alone, the same pose three times in a batch of five, and the same call again: identical bits (the grid's
    atomicAdd fill order and the other poses' clusters must not leak into a result)"""
    model, scene, start = case_synth(2049, 1500)
    _, _, other = case_synth(2049, 1500, k=1)
    dm, ds = ctx.upload_cloud(model), ctx.upload_cloud(scene)
    P1, r1, it1 = ctx.icp_refine(dm, ds, start[None], 3, 0.0, 2.5, 2)
    P2, r2, it2 = ctx.icp_refine(dm, ds, start[None], 3, 0.0, 2.5, 2)
    batch = np.stack([start, other, start, np.eye(4), start])
    PB, rB, itB = ctx.icp_refine(dm, ds, batch, 3, 0.0, 2.5, 2)
    assert np.array_equal(P1, P2) and np.array_equal(r1, r2) and it1 == it2
    for k in (0, 2, 4):
        assert np.array_equal(PB[k], P1[0]) and rB[k] == r1[0], k
    assert itB >= 3 * it1
