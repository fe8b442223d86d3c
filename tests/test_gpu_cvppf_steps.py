"""K7 (k7_cvppf.cu, b200cv_*) against the float64 NumPy restatement of PPF3DDetector (tests/cvppf_reference.py) and,
where it has a hook, the CPU oracle: every reference point, past one reference per CTA, across the sampling step, the
number of angles, the scene step and distance, match_S2B, the search parameters and crafted edges.

Each case first asserts that no decision of the restatement (keys, alpha indices, float(alpha), pose branches, cluster
thresholds) sits within a last-bit difference of an edge; then training is compared bit for bit (sampled model, every
offset and node of the table, the whole alpha_m matrix), every reference's peak triple exactly and its pose, angle, t
and q within 1e-12, accumulators bit for bit at the references where the persistent voting loop changes hands (r = 0,
grid - 1, grid, grid + 1, 2 grid + 1, the last and four seeded random ones), and every pose cluster (votes, leader,
pose within 1e-9).  What may differ is only libm's last ulp in sin / cos / acos / atan2.
"""
import numpy as np
import pytest

import cvppf_reference as cr

pytestmark = pytest.mark.gpu

RAW_TOL = 1e-12
CLUSTER_TOL = 1e-9


def _grid(refs):
    import torch
    return min(refs, 2 * torch.cuda.get_device_properties(0).multi_processor_count)


def _acc_refs(refs, grid, extra=()):
    picks = {0, grid - 1, grid, grid + 1, 2 * grid + 1, refs - 1} | set(int(r) for r in extra)
    picks |= set(np.random.default_rng(4).choice(refs, min(4, refs), replace=False).tolist())
    return sorted(r for r in picks if 0 <= r < refs)


def _close_pose(a, b, extent, tol):
    """rotation entries absolutely, translations relative to the scene's extent"""
    a, b = a.reshape(-1, 4, 4), b.reshape(-1, 4, 4)
    return max(np.abs(a[:, :3, :3] - b[:, :3, :3]).max(initial=0.0),
               np.abs(a[:, :3, 3] - b[:, :3, 3]).max(initial=0.0) / extent)


def run_case(ctx, oracle, name, model, scene, ss, na, sstep, sd, edge=None, pos=None, rot=None, past_one_ref=False):
    from yolo_ppf_pose_estimation_b200 import capi
    tr = cr.train(model, ss, na)
    assert tr.margins.unsafe() == 0, tr.margins.report()
    dev = capi.CvDetector(ctx, ss, 0.05, na).train_model(model)
    ref = oracle.CvDetector(ss, 0.05, na).train_model(model)
    if pos is not None or rot is not None:
        dev.set_search_params(-1 if pos is None else pos, -1 if rot is None else rot)
        ref.set_search_params(-1 if pos is None else pos, -1 if rot is None else rot)
    # training
    ci = dev.info
    m = tr.m
    assert ci.n_sampled == m and ci.table_size == tr.table_size and ci.n_nodes == m * (m - 1)
    assert ci.num_angles == tr.num_angles and ci.angle_step == tr.angle_step and ci.distance_step == tr.distance_step
    assert np.array_equal(dev.model_points().view(np.uint32), tr.model.view(np.uint32))
    off, nodes, alpha = dev.table_export()
    assert np.array_equal(off, tr.offsets) and np.array_equal(nodes, tr.nodes)
    assert np.array_equal(alpha.view(np.uint32), tr.alpha_m.view(np.uint32))
    # per reference
    step = int(1.0 / sstep)
    refs = (len(cr.sample(scene, np.float32(sd))) + step - 1) // step
    grid = _grid(refs)
    if past_one_ref:
        assert refs > grid, (refs, grid)
    mt0 = cr.match(tr, scene, sstep, sd, edge=edge, position_threshold=pos, rotation_threshold=rot)
    picks = _acc_refs(refs, grid, mt0.overflow_refs[:4])
    mt = cr.match(tr, scene, sstep, sd, edge=edge, position_threshold=pos, rotation_threshold=rot, keep_accumulators=picks)
    assert mt.refs == refs and mt.margins.unsafe() == 0, mt.margins.report()
    res, ncl = dev.match(scene, sstep, sd, max_poses=refs) if edge is None else dev.match_s2b(scene, edge, sstep, sd, max_poses=refs)
    assert np.array_equal(dev.scene_points().view(np.uint32), mt.scene.view(np.uint32))
    assert dev.info.n_scene_sampled == len(mt.scene) and dev.info.n_second_sampled == len(mt.second)
    raw = dev.raw_poses()
    assert len(raw) == refs
    for f in ("num_votes", "model_index", "alpha_index", "reference_index"):
        assert np.array_equal(raw[f], mt.raw[f]), f
    assert np.array_equal(raw["alpha"], mt.raw["alpha"])
    lo, hi = cr.bbox(scene)
    extent = max(1.0, float(np.linalg.norm(hi.astype(np.float64) - lo)))
    assert _close_pose(raw["pose"], mt.raw["pose"], extent, RAW_TOL) < RAW_TOL
    assert np.abs(raw["angle"] - mt.raw["angle"]).max() < RAW_TOL
    assert np.abs(raw["t"] - mt.raw["t"]).max() / extent < RAW_TOL
    assert np.abs(raw["q"] - mt.raw["q"]).max() < RAW_TOL
    # the oracle's peaks and clusters
    if edge is None:
        rposes, rvotes, rraw, rncl = ref.match(scene, sstep, sd, max_poses=refs)
    else:
        rposes, rvotes, rraw, rncl = ref.match_s2b(scene, edge, sstep, sd, max_poses=refs)
    assert np.array_equal(rraw[:, 0], raw["num_votes"]) and np.array_equal(rraw[:, 1], raw["model_index"])
    assert np.array_equal(rraw[:, 2], raw["alpha_index"])
    # clusters
    assert ncl == len(mt.clusters) == rncl and len(res) == ncl
    want = mt.clusters
    assert np.array_equal(res["num_votes"], [c["num_votes"] for c in want]) and np.array_equal(res["num_votes"], rvotes)
    leaders = np.array([c["leader"] for c in want])
    assert np.array_equal(res["reference_index"], leaders)
    assert np.array_equal(res["model_index"], mt.raw["model_index"][leaders])
    assert np.array_equal(res["alpha_index"], mt.raw["alpha_index"][leaders])
    assert _close_pose(res["pose"], np.stack([c["pose"] for c in want]), extent, CLUSTER_TOL) < CLUSTER_TOL
    assert _close_pose(res["pose"], rposes, extent, CLUSTER_TOL) < CLUSTER_TOL
    # accumulators where the persistent loop changes hands (each call votes every reference again)
    for r in picks:
        acc = dev.accumulator(scene, r, sstep, sd, edge=edge)
        assert np.array_equal(acc, mt.accumulators[r]), r
    print(f"CASE {name}: m {m} refs {refs} grid {grid} clusters {ncl} compared {ncl} accumulators {picks} "
          f"unsafe {tr.margins.unsafe() + mt.margins.unsafe()} ties {mt.ties} overflow {mt.overflow}")
    return dev, tr, mt, res, raw


@pytest.fixture(scope="module")
def bottle_case(bottle_5mm):
    return cr.bottle_scene(bottle_5mm)


def test_baseline(ctx, oracle, bottle_case):
    """today's configuration: sampling 0.04, 30 angles, scene step 1/5, distance 0.04; the rigid motion is recovered"""
    model, scene, edge, G = bottle_case
    dev, tr, mt, res, raw = run_case(ctx, oracle, "baseline", model, scene, 0.04, 30, 1.0 / 5.0, 0.04)
    assert dev.info.num_angles == 30
    P = res["pose"][0].reshape(4, 4)
    pts = model[:, :3].astype(np.float64)
    err = np.linalg.norm((pts @ P[:3, :3].T + P[:3, 3]) - (pts @ G[:3, :3].T + G[:3, 3]), axis=1).mean()
    assert err < 0.02, err


@pytest.mark.parametrize("name,ss,na,sstep,sd", [
    ("multi-ref", 0.04, 30, 1.0, 0.02),
    ("big model", 0.025, 30, 1.0, 0.02),
    ("small model", 0.1, 30, 1.0 / 2.0, 0.02),
    ("angles 13", 0.04, 13, 1.0, 0.04),
    ("angles 7", 0.04, 7, 1.0 / 2.0, 0.04),
    ("angles 360", 0.04, 360, 1.0 / 2.0, 0.04),
])
def test_parameters(ctx, oracle, bottle_case, name, ss, na, sstep, sd):
    model, scene, edge, G = bottle_case
    dev, tr, mt, res, raw = run_case(ctx, oracle, name, model, scene, ss, na, sstep, sd, past_one_ref=name == "multi-ref")
    if na == 13:
        assert dev.info.num_angles == 12  # floor(2 pi / (2 pi / 13)): upstream's numAngles


def test_s2b(ctx, oracle, bottle_case):
    """match_S2B: references from the surface cloud, paired with the sampled edge cloud"""
    model, scene, edge, G = bottle_case
    dev, tr, mt, res, raw = run_case(ctx, oracle, "S2B", model, scene, 0.04, 30, 1.0, 0.02, edge=edge)
    assert dev.info.n_second_sampled == len(oracle.cv_sample(edge, 0.02)) < dev.info.n_scene_sampled


def test_long_loop(ctx, oracle, bottle_5mm):
    """denser clutter: every CTA votes for more than four references"""
    model, scene, edge, G = cr.bottle_scene(bottle_5mm, n_clutter=3000, seed=8)
    dev, tr, mt, res, raw = run_case(ctx, oracle, "long loop", model, scene, 0.04, 30, 1.0, 0.02, past_one_ref=True)
    assert mt.refs > 4 * _grid(mt.refs)


def test_position_threshold_zero(ctx, oracle, bottle_case):
    """every pose its own cluster: the clusters are the poses by votes descending, ties in reference order"""
    model, scene, edge, G = bottle_case
    dev, tr, mt, res, raw = run_case(ctx, oracle, "threshold 0", model, scene, 0.04, 30, 1.0, 0.02, pos=0.0, past_one_ref=True)
    assert len(res) == mt.refs
    order = np.argsort(-raw["num_votes"].astype(np.int64), kind="stable")
    assert np.array_equal(res["reference_index"], order) and np.array_equal(res["num_votes"], raw["num_votes"][order])
    assert (np.diff(raw["num_votes"][order].astype(np.int64)) < 0).sum() < mt.refs - 1  # ties exist and are ordered


def test_huge_threshold(ctx, oracle, bottle_case):
    """one cluster holding every vote"""
    model, scene, edge, G = bottle_case
    dev, tr, mt, res, raw = run_case(ctx, oracle, "huge threshold", model, scene, 0.04, 30, 1.0, 0.02, pos=1e3, rot=10.0,
                                     past_one_ref=True)
    assert len(res) == 1 and res["num_votes"][0] == raw["num_votes"].sum()


@pytest.mark.parametrize("num_angles", [30, 13])
def test_alpha_index_overflow_into_the_next_row(ctx, oracle, num_angles):
    """alpha index numAngles: bin 0 of the next model point's row, dropped on the last row (upstream's arithmetic)"""
    model, scene = cr.lattice_overflow()
    dev, tr, mt, res, raw = run_case(ctx, oracle, f"overflow {num_angles}", model, scene, cr.LATTICE_STEP, num_angles, 1.0,
                                     cr.LATTICE_STEP)
    assert mt.overflow["before_last_row"] >= 1 and mt.overflow["last_row"] >= 1, mt.overflow
    assert mt.overflow_refs  # their accumulators were compared above


def test_tie_at_the_peak(ctx, oracle):
    model, scene = cr.symmetric_tie()
    dev, tr, mt, res, raw = run_case(ctx, oracle, "tie", model, scene, 0.05, 30, 1.0, 0.05)
    assert mt.ties >= 1


def test_zero_normal(ctx, oracle):
    model, scene = cr.lattice_overflow(zero_normal=True)
    dev, tr, mt, res, raw = run_case(ctx, oracle, "zero normal", model, scene, cr.LATTICE_STEP, 30, 1.0, cr.LATTICE_STEP)
    assert np.count_nonzero(~dev.model_points()[:, 3:].any(axis=1)) == 1


def test_model_past_the_table_limit_is_refused(ctx, oracle, bottle_case):
    """more than 46340 sampled points (m^2 > 2^31) would need a 2^32-bucket table: refused before any table memory, and the
    detector trains and matches afterwards"""
    from yolo_ppf_pose_estimation_b200 import capi
    cloud = cr.over_limit_cloud()
    assert len(cr.sample(cloud, np.float32(0.01))) > cr.TABLE_MAX_POINTS
    dev = capi.CvDetector(ctx, 0.01, 0.05)
    with pytest.raises(capi.B200PPFError) as e:
        dev.train_model(cloud)
    assert e.value.code == -5  # B200PPF_ERR_UNSUPPORTED
    with pytest.raises(capi.B200PPFError):
        dev.match(bottle_case[1])  # not trained
    model, scene, edge, G = bottle_case
    dev.train_model(model)  # the same detector: 0.01 keeps the bottle far below the limit
    tr = cr.train(model, 0.01, 30)
    assert dev.info.n_sampled == tr.m and np.array_equal(dev.model_points().view(np.uint32), tr.model.view(np.uint32))
    res, ncl = dev.match(scene, 1.0 / 5.0, 0.04)
    _, rvotes, rraw, rncl = oracle.CvDetector(0.01, 0.05).train_model(model).match(scene, 1.0 / 5.0, 0.04)
    assert ncl == rncl >= 1 and np.array_equal(dev.raw_poses()["num_votes"], rraw[:, 0])
    assert np.array_equal(res["num_votes"], rvotes)
