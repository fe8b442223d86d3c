"""CPU tests of oracle/cvppf_oracle.cpp — the restatement of cv::ppf_match_3d::PPF3DDetector, the engine the reference
actually calls (include/CloudProcessing.h:205-236, :442).  It is the checker of a row that is not built on the device
yet (SURVEY.md §8f rank 4); these tests pin what can be pinned offline: the hash against published MurmurHash3 vectors,
the sampling and the pair feature against numpy restatements, and the whole train / match / cluster chain against a
known rigid motion.  The rest of the chain is compared with tests/cvppf_reference.py in test_cvppf_reference_host.py."""
import struct

import numpy as np
import pytest

import cvppf_reference as cr


def test_murmur3_x86_32_known_answers(oracle):
    # the vectors commonly used to validate MurmurHash3_x86_32 implementations
    assert oracle.cv_murmur(b"", 0) == 0
    assert oracle.cv_murmur(b"", 1) == 0x514E28B7
    assert oracle.cv_murmur(b"", 0xFFFFFFFF) == 0x81F16F39
    assert oracle.cv_murmur(b"\xff\xff\xff\xff", 0) == 0x76293B50
    assert oracle.cv_murmur(b"\x21\x43\x65\x87", 0) == 0xF55B516B
    assert oracle.cv_murmur(b"\x21\x43\x65\x87", 0x5082EDEE) == 0x2362F9DE
    assert oracle.cv_murmur(b"\x21\x43\x65", 0) == 0x7E4A8634
    assert oracle.cv_murmur(b"\x21\x43", 0) == 0xA0F7B07A
    assert oracle.cv_murmur(b"\x21", 0) == 0x72661CF4
    assert oracle.cv_murmur(b"\x00\x00\x00\x00", 0) == 0x2362F9DE


def test_pair_feature_and_hash(oracle, bottle_5mm):
    a_step, d_step = 2 * np.pi / 30, 0.01
    rng = np.random.default_rng(0)
    for i, j in rng.integers(0, bottle_5mm.shape[0], (200, 2)):
        f, h = oracle.cv_pair(bottle_5mm[i], bottle_5mm[j], a_step, d_step)
        p1, n1, p2, n2 = (bottle_5mm[i, :3].astype(np.float64), bottle_5mm[i, 3:].astype(np.float64),
                          bottle_5mm[j, :3].astype(np.float64), bottle_5mm[j, 3:].astype(np.float64))
        d = p2 - p1
        if np.linalg.norm(d) <= 1.192092896e-07:
            assert not f.any()
            continue
        dn = d / np.linalg.norm(d)
        ang = lambda a, b: np.arctan2(np.linalg.norm(np.cross(a, b)), a @ b)
        ref = np.array([ang(n1, dn), ang(n2, dn), ang(n1, n2), np.linalg.norm(d)])
        assert np.abs(f - ref).max() < 1e-12
        key = struct.pack("<4i", int(f[0] / a_step), int(f[1] / a_step), int(f[2] / a_step), int(f[3] / d_step))
        assert h == oracle.cv_murmur(key, 42)


def test_sample_by_quantization(oracle, bottle_5mm):
    """float32 cell arithmetic, upstream's stride ns (a coordinate on the upper bound shares a neighbour's list), averages
    in double in input order: the restatement in tests/cvppf_reference.py and the oracle agree bit for bit"""
    assert int(1.0 / float(np.float32(0.05))) == 19  # (int)(1.0 / sampleStep) with a float step: 19 cells, not 20
    for step in (0.05, 0.04, 0.1, 1.0 / 8.5):
        out = cr.sample(bottle_5mm, np.float32(step))
        assert np.array_equal(out.view(np.uint32), oracle.cv_sample(bottle_5mm, step).view(np.uint32)), step
        assert 100 < out.shape[0] < bottle_5mm.shape[0]
        assert np.abs(np.linalg.norm(out[:, 3:], axis=1) - 1).max() < 1e-6
        index, ns = cr.sample_cells(bottle_5mm, np.float32(step))
        assert index.max() >= ns * ns * ns  # the points on the upper bound of x exist and land past the last full cell


def _rigid(axis, angle, t):
    axis = np.asarray(axis, np.float64) / np.linalg.norm(axis)
    K = np.array([[0, -axis[2], axis[1]], [axis[2], 0, -axis[0]], [-axis[1], axis[0], 0]])
    T = np.eye(4)
    T[:3, :3] = np.eye(3) + np.sin(angle) * K + (1 - np.cos(angle)) * K @ K
    T[:3, 3] = t
    return T


# rotations with a positive trace: beyond 120 degrees the cluster average adds quaternions from different branches of the
# matrix -> quaternion conversion without aligning their signs (upstream does the same), and which poses flip depends on a
# convention this restatement cannot pin (see the header of cvppf_oracle.cpp)
@pytest.mark.parametrize("angle,t", [(0.7, (0.1, -0.05, 0.3)), (1.3, (-0.3, 0.2, 0.1))])
def test_train_match_recovers_a_rigid_motion(oracle, bottle_5mm, angle, t):
    det = oracle.CvDetector(0.04, 0.05).train_model(bottle_5mm)
    m = det.model_points()
    assert 300 < det.n_model == m.shape[0] < bottle_5mm.shape[0]
    G = _rigid((0.3, 1.0, 0.2), angle, t)
    rng = np.random.default_rng(7)
    inst = np.concatenate([bottle_5mm[:, :3] @ G[:3, :3].T + G[:3, 3], bottle_5mm[:, 3:] @ G[:3, :3].T], axis=1)
    centre = inst[:, :3].mean(0)
    clutter = np.concatenate([centre + rng.normal(scale=0.15, size=(600, 3)), rng.normal(size=(600, 3))], axis=1)
    clutter[:, 3:] /= np.linalg.norm(clutter[:, 3:], axis=1, keepdims=True)
    scene = np.concatenate([inst, clutter]).astype(np.float32)
    poses, votes, raw, n_clusters = det.match(scene, 1.0 / 5.0, 0.04)
    assert n_clusters >= 1 and votes[0] == votes.max() and raw[:, 0].max() > 0
    P = poses[0]
    assert np.abs(P[:3, :3] @ P[:3, :3].T - np.eye(3)).max() < 1e-9 and np.isclose(np.linalg.det(P[:3, :3]), 1.0)
    dR = P[:3, :3].T @ G[:3, :3]
    rot_err = np.degrees(np.arccos(np.clip((np.trace(dR) - 1) / 2, -1, 1)))
    # the model's own points mapped by the two poses (the translation alone is dominated by the lever arm to the origin)
    pts = bottle_5mm[:, :3].astype(np.float64)
    err = np.linalg.norm((pts @ P[:3, :3].T + P[:3, 3]) - (pts @ G[:3, :3].T + G[:3, 3]), axis=1).mean()
    print(f"angle {angle}: {n_clusters} clusters, votes {votes[:3].tolist()}, rotation error {rot_err:.2f} deg, mean point error {1e3 * err:.1f} mm")
    # the bottle is nearly a surface of revolution: the angle about its own axis is weakly determined, so the bars are
    # the direction of that axis (one alpha bin) and the mean point error (a tenth of the diameter), before any ICP
    axis = np.linalg.eigh(np.cov((pts - pts.mean(0)).T))[1][:, -1]
    axis_err = np.degrees(np.arccos(np.clip(abs((P[:3, :3] @ axis) @ (G[:3, :3] @ axis)), -1, 1)))
    print(f"   axis error {axis_err:.2f} deg")
    assert axis_err < 12.0 and err < 0.02 and rot_err < 30.0
    # threads do not change anything
    poses1, votes1, raw1, _ = det.match(scene, 1.0 / 5.0, 0.04, n_threads=1)
    assert np.array_equal(poses, poses1) and np.array_equal(votes, votes1) and np.array_equal(raw, raw1)


def test_parity_hooks_agree_with_match(oracle, bottle_5mm):
    """The hooks the device engine's tests use (bucket contents, one reference point's accumulator, match_S2B as inferred)
    are consistent with match() itself: the peak of every sampled accumulator is the raw pose of that reference point."""
    det = oracle.CvDetector(0.05, 0.05).train_model(bottle_5mm)
    m = det.n_model
    assert det.table_size >= m * m and det.table_size & (det.table_size - 1) == 0
    total = 0
    for b in range(0, det.table_size, max(1, det.table_size // 4096)):
        nodes = det.bucket(b)
        assert (np.diff(nodes.astype(np.int64)) > 0).all() and (nodes // m != nodes % m).all()
        total += len(nodes)
    assert total > 0
    scene = bottle_5mm[::2].copy()
    poses, votes, raw, ncl = det.match(scene, 1.0 / 5.0, 0.05)
    for r in (0, len(raw) // 2, len(raw) - 1):
        acc = det.accumulator(scene, r * 5, 0.05)
        flat = int(np.argmax(acc))
        assert raw[r, 0] == acc.reshape(-1)[flat] and (int(raw[r, 1]), int(raw[r, 2])) == divmod(flat, acc.shape[1])
    # match_S2B with a thin "edge" cloud: fewer pairs per reference point, never more votes than the surface pairing casts
    edge = scene[::7].copy()
    p2, v2, raw2, ncl2 = det.match_s2b(scene, edge, 1.0 / 5.0, 0.05)
    assert len(raw2) == len(raw) and raw2[:, 0].sum() < raw[:, 0].sum() and ncl2 >= 1
    acc = det.accumulator(scene, 10, 0.05, edge=edge)
    assert raw2[2, 0] == acc.max()
