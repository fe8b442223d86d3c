"""The float64 NumPy restatement of PPF3DDetector (tests/cvppf_reference.py) against the CPU oracle
(oracle/cvppf_oracle.cpp): two independent statements of upstream's trainModel / match / clusterPoses must agree bit
for bit on everything integer (sampled clouds, buckets, accumulators, peaks, cluster votes) and to rounding on poses.
Every case first asserts that none of the restatement's decisions sits on an edge (see that module's header)."""
import numpy as np
import pytest

import cvppf_reference as cr

# (sampling step, numAngles asked for, relative scene sample step, relative scene distance)
PARAMS = {"baseline": (0.04, 30, 1.0 / 5.0, 0.04), "small model, 13 angles": (0.1, 13, 1.0 / 2.0, 0.04)}


def test_murmur_matches_the_oracle(oracle):
    rng = np.random.default_rng(1)
    for words in (1, 2, 4):
        keys = rng.integers(-2 ** 31, 2 ** 31, (300, words)).astype(np.int32)
        keys[:4] = [[0] * words, [-1] * words, [1] * words, [2 ** 31 - 1] * words]
        got = cr.murmur3_x86_32(keys)
        for k, h in zip(keys, got):
            assert int(h) == oracle.cv_murmur(k.tobytes(), 42)
    seeded = cr.murmur3_x86_32(np.array([[0x87654321]], np.uint32), seed=0x5082EDEE)
    assert int(seeded[0]) == 0x2362F9DE  # a published MurmurHash3_x86_32 vector


def _check_case(oracle, model, scene, ss, na, sstep, sd, acc_refs=10, edge=None):
    tr = cr.train(model, ss, na)
    assert tr.margins.unsafe() == 0, tr.margins.report()
    ref = oracle.CvDetector(ss, 0.05, na).train_model(model)
    assert np.array_equal(tr.model.view(np.uint32), ref.model_points().view(np.uint32))
    assert ref.num_angles == tr.num_angles == int(np.floor(2 * np.pi / tr.angle_step))
    off, nodes = ref.table_export()
    assert ref.table_size == tr.table_size and np.array_equal(off, tr.offsets) and np.array_equal(nodes, tr.nodes)
    first = cr.match(tr, scene, sstep, sd, edge=edge)
    refs = first.refs
    picks = sorted(set(np.random.default_rng(2).choice(refs, min(acc_refs, refs), replace=False).tolist()) |
                   set(first.overflow_refs))
    mt = cr.match(tr, scene, sstep, sd, edge=edge, keep_accumulators=picks)
    assert mt.margins.unsafe() == 0, mt.margins.report()
    if edge is None:
        poses, votes, raw, ncl = ref.match(scene, sstep, sd, max_poses=refs)
    else:
        poses, votes, raw, ncl = ref.match_s2b(scene, edge, sstep, sd, max_poses=refs)
    assert raw.shape[0] == refs
    assert np.array_equal(raw[:, 0], mt.raw["num_votes"]) and np.array_equal(raw[:, 1], mt.raw["model_index"])
    assert np.array_equal(raw[:, 2], mt.raw["alpha_index"])
    for r in picks:
        assert np.array_equal(ref.accumulator(scene, r * mt.step, sd, edge=edge), mt.accumulators[r]), r
    assert ncl == len(mt.clusters)
    assert np.array_equal(votes, [c["num_votes"] for c in mt.clusters])
    assert np.abs(poses - np.stack([c["pose"] for c in mt.clusters])).max() < 1e-12
    return tr, mt


@pytest.mark.parametrize("name", list(PARAMS))
def test_restatement_matches_the_oracle(oracle, bottle_5mm, name):
    model, scene, edge, G = cr.bottle_scene(bottle_5mm)
    tr, mt = _check_case(oracle, model, scene, *PARAMS[name])
    if name == "baseline":
        P = mt.clusters[0]["pose"]
        pts = model[:, :3].astype(np.float64)
        err = np.linalg.norm((pts @ P[:3, :3].T + P[:3, 3]) - (pts @ G[:3, :3].T + G[:3, 3]), axis=1).mean()
        assert err < 0.02, err
    else:
        assert tr.num_angles == 12  # floor(2 pi / (2 pi / 13)) = 12: one bin fewer than asked, as upstream


def test_s2b_restatement_matches_the_oracle(oracle, bottle_5mm):
    model, scene, edge, G = cr.bottle_scene(bottle_5mm)
    _check_case(oracle, model, scene, 0.04, 30, 1.0 / 5.0, 0.04, acc_refs=4, edge=edge)


@pytest.mark.parametrize("num_angles", [30, 13])
def test_alpha_index_overflow_into_the_next_row(oracle, num_angles):
    """alpha_m = float(pi) against alpha_s = -pi + 1.5e-8: index numAngles, counted in bin 0 of the next model point's
    row, dropped on the last row — upstream's arithmetic, on both sides"""
    model, scene = cr.lattice_overflow()
    assert len(cr.sample(model, np.float32(cr.LATTICE_STEP))) == len(model)  # one point per cell
    tr, mt = _check_case(oracle, model, scene, cr.LATTICE_STEP, num_angles, 1.0, cr.LATTICE_STEP, acc_refs=4)
    assert mt.overflow["before_last_row"] >= 1 and mt.overflow["last_row"] >= 1, mt.overflow
    assert tr.num_angles == (30 if num_angles == 30 else 12)


def test_tie_at_the_peak(oracle):
    """a quarter-turn-symmetric cloud: some reference's maximum occurs more than once, and the first one in
    (model point, alpha index) order is the peak"""
    model, scene = cr.symmetric_tie()
    tr, mt = _check_case(oracle, model, scene, 0.05, 30, 1.0, 0.05, acc_refs=4)
    assert mt.ties >= 1


def test_zero_normal(oracle):
    """two points with opposite normals in one cell sample to a point whose normal is (0, 0, 0)"""
    model, scene = cr.lattice_overflow(zero_normal=True)
    sampled = cr.sample(model, np.float32(cr.LATTICE_STEP))
    assert np.count_nonzero(~sampled[:, 3:].any(axis=1)) == 1
    _check_case(oracle, model, scene, cr.LATTICE_STEP, 30, 1.0, cr.LATTICE_STEP, acc_refs=4)


def test_over_limit_cloud_samples_past_the_table_limit():
    cloud = cr.over_limit_cloud()
    assert len(cr.sample(cloud, np.float32(0.01))) > cr.TABLE_MAX_POINTS
    assert cr.TABLE_MAX_POINTS ** 2 <= 2 ** 31 < (cr.TABLE_MAX_POINTS + 1) ** 2
