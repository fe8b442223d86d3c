"""The NumPy restatement of the ICP (tests/icp_reference.py) against the CPU oracle, and the oracle's 6 x 6 solve against
np.linalg.pinv.  CPU only: these pin the yardstick that tests/test_gpu_icp_steps.py holds the device to."""
import numpy as np
import pytest

import icp_reference as ir


def _rot(axis, ang):
    axis = np.asarray(axis, np.float64) / np.linalg.norm(axis)
    K = np.array([[0, -axis[2], axis[1]], [axis[2], 0, -axis[0]], [-axis[1], axis[0], 0]])
    return np.eye(3) + np.sin(ang) * K + (1 - np.cos(ang)) * K @ K


@pytest.fixture(scope="module")
def synth_case():
    """1 500-point synthetic bottle, its 2 000-point neighbourhood of the synthetic scene, a start 6 degrees / 1 cm off"""
    from yolo_ppf_pose_estimation_b200 import synth
    model = synth.synth_model(1500, 1)
    G = synth.gt_pose(2)
    sc = synth.synth_scene(20000, 2, model_seed=1)
    centre = G[:3, 3] + G[:3, :3] @ np.array([0.0, 0.0, 0.09])
    scene = sc[np.linalg.norm(sc[:, :3] - centre, axis=1) < 0.2]
    D = np.eye(4)
    D[:3, :3] = _rot([0.3, 1.0, 0.2], 0.1)
    D[:3, 3] = (0.01, -0.005, 0.003)
    return model, scene, D @ G


def _assert_same(res, R, rres, rit):
    assert res.iterations == rit
    scale = max(1.0, np.abs(R).max())
    assert np.abs(res.pose - R).max() <= 1e-11 * scale, np.abs(res.pose - R).max()
    assert abs(res.residual - rres) <= 1e-11 * max(1.0, abs(rres))


@pytest.mark.parametrize("levels", [1, 2, 3])
@pytest.mark.parametrize("iterations", [1, 2, 3, 4, 5, 6])
def test_restatement_equals_oracle(oracle, synth_case, levels, iterations):
    """tolerance 0: every level runs exactly round(iterations / (L+1)) iterations, on both sides"""
    model, scene, start = synth_case
    res = ir.register(model, scene, start, iterations, 0.0, 2.5, levels)
    R, rres, rit = oracle.icp_refine(model, scene, start[None], iterations, 0.0, 2.5, levels)
    _assert_same(res, R[0], rres[0], rit)
    assert res.iterations == sum(int(np.rint(iterations / (L + 1))) for L in range(levels))
    assert [t.level for t in res.trace] == sorted((t.level for t in res.trace), reverse=True)


def test_restatement_equals_oracle_with_the_stop_test_and_without_rejection(oracle, synth_case):
    model, scene, start = synth_case
    for kw in (dict(max_iterations=40, tolerance=0.005, rejection_scale=2.5, num_levels=3),
               dict(max_iterations=6, tolerance=0.0, rejection_scale=0.0, num_levels=2)):
        res = ir.register(model, scene, start, **kw)
        R, rres, rit = oracle.icp_refine(model, scene, start[None], **kw)
        _assert_same(res, R[0], rres[0], rit)
    assert all(t.threshold == np.inf for t in res.trace)


def test_restatement_equals_oracle_on_the_reference_object(oracle, oracle_bottle, bottle, scene_crop):
    """The 543-point bottle over 8 levels keeps 4 model samples at the coarsest: the minimum-norm branch runs"""
    _, hm = oracle_bottle
    _, poses, _, _ = hm.register(bottle, scene_crop, ref_rate=5, n_threads=4)
    start = poses[0].astype(np.float64)
    res = ir.register(bottle, scene_crop, start, 16, 0.0, 2.5, 8)
    R, rres, rit = oracle.icp_refine(bottle, scene_crop, start[None], 16, 0.0, 2.5, 8)
    _assert_same(res, R[0], rres[0], rit)
    assert "min_norm" in [t.branch for t in res.trace] and "elimination" in [t.branch for t in res.trace]


def _gram(rank, seed, n_rows=40):
    rng = np.random.default_rng(seed)
    A = rng.normal(size=(n_rows, rank)) @ rng.normal(size=(rank, 6))
    b = rng.normal(size=n_rows)
    return A.T @ A, A.T @ b, A, b


@pytest.mark.parametrize("rank", [1, 2, 3, 4, 5, 6])
def test_solve6_is_the_minimum_norm_least_squares_solution(oracle, rank):
    """rank 1 to 6: the pseudo-inverse solution of the n x 6 system, and the restatement's solve to the last bit"""
    for seed in range(3):
        N, g, A, b = _gram(rank, 10 * rank + seed)
        x = oracle.solve6(N, g)
        want = np.linalg.pinv(A, rcond=1e-10) @ b
        assert np.allclose(x, want, rtol=1e-8, atol=1e-9 * np.abs(want).max()), (rank, seed, x, want)
        xr, branch, _, _ = ir.solve6(N, g)
        assert branch == ("elimination" if rank == 6 else "min_norm")
        assert np.array_equal(xr, x)


@pytest.mark.parametrize("side", [1.01, 0.99])
def test_solve6_at_the_eigenvalue_cut(oracle, side):
    """rank 5 plus a sixth eigenvalue 1 % above / below 1e-12 of the largest: kept above the cut, dropped below it"""
    rng = np.random.default_rng(7)
    Q, _ = np.linalg.qr(rng.normal(size=(6, 6)))
    lam = np.array([4.0, 2.0, 1.0, 0.5, 0.25, 4.0 * 1e-12 * side])
    N = (Q * lam) @ Q.T
    N = 0.5 * (N + N.T)
    x_true = Q @ np.array([1.0, -2.0, 0.5, 3.0, -1.0, 1.0])   # unit component along the weak direction
    g = N @ x_true
    x = oracle.solve6(N, g)
    xr, branch, _, eig_margin = ir.solve6(N, g)
    assert branch == "min_norm" and np.array_equal(xr, x)
    assert 0.005 < eig_margin < 0.02                           # the weak eigenvalue, 1 % from the cut
    w, V = np.linalg.eigh(N)
    keep = w > 1e-12 * w.max()
    assert keep.sum() == (6 if side > 1 else 5)
    want = (V[:, keep] / w[keep]) @ (V[:, keep].T @ g)
    weak = Q[:, 5] @ x
    if side > 1:
        assert abs(weak - 1.0) < 1e-3, weak                   # 1e-16 of noise in g over a 4e-12 eigenvalue
        assert np.allclose(x, want, rtol=0, atol=1e-3)
    else:
        assert abs(weak) < 1e-9, weak
        assert np.allclose(x, want, rtol=1e-9, atol=1e-12)
        assert np.allclose(x, x_true - Q[:, 5], rtol=1e-9, atol=1e-12)
