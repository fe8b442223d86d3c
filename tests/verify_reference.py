"""Float64 restatement of b200ppf_score_poses (include/b200ppf.h, pose verification), with numpy and scipy's kd-tree.

For a model (N, 6), a scene (M, 6) and a pose T (model -> scene): model point p with normal n moves to p' = R p + t,
n' = R n; it is visible when n'.(-p') > 0 or n is zero; a visible point is an inlier when its nearest scene point q (the
lowest index among equally near ones) lies within inlier_dist and n_q.n' >= cos(normal_angle) (no normal test when
normal_angle >= pi).  The parameters are taken as the float32 values the library receives.

score() also returns the borderline points, whose outcome may differ from the device's by rounding: a distance within
1e-5 * inlier_dist of inlier_dist, a visibility or normal dot product within 1e-6 of its bound, or a second scene point as
near as the nearest within 1e-6 relative."""
import numpy as np
from scipy.spatial import cKDTree

DIST_TOL, DOT_TOL, TIE_TOL = 1e-5, 1e-6, 1e-6


def score(model, scene, pose, inlier_dist=0.01, normal_angle=np.radians(30.0)):
    """-> dict(inliers, visible, fit, rms, inlier (N,) bool, visible_mask (N,) bool, borderline (N,) bool)"""
    model = np.asarray(model, np.float32)
    scene = np.asarray(scene, np.float32).reshape(-1, 6)
    T = np.asarray(pose, np.float64).reshape(4, 4)
    tau = float(np.float32(inlier_dist))
    use_normals = not (np.float32(normal_angle) >= np.float32(np.pi))
    cos_min = float(np.cos(np.float64(np.float32(normal_angle))))
    m = model.astype(np.float64)
    p = m[:, :3] @ T[:3, :3].T + T[:3, 3]
    n = m[:, 3:6] @ T[:3, :3].T
    zero = np.all(model[:, 3:6] == 0, axis=1)
    vdot = -np.einsum("ij,ij->i", n, p)
    visible = zero | (vdot > 0)
    border = ~zero & (np.abs(vdot) <= DOT_TOL)
    inlier = np.zeros(len(model), bool)
    d0 = np.full(len(model), np.inf)
    if len(scene) and len(model):
        s = scene[:, :3].astype(np.float64)
        k = min(3, len(scene))
        d, j = cKDTree(s).query(p, k=k)
        d, j = d.reshape(len(p), k), j.reshape(len(p), k)
        # exact distances, the lowest index among the equally near
        dd = np.sqrt(((s[j] - p[:, None, :]) ** 2).sum(-1))
        order = np.lexsort((j, dd))  # per row: by distance, then index
        rows = np.arange(len(p))[:, None]
        dd, j = dd[rows, order], j[rows, order]
        d0 = dd[:, 0]
        q = j[:, 0]
        near = d0 <= tau
        ndot = np.einsum("ij,ij->i", scene[q, 3:6].astype(np.float64), n)
        ok = near & ((not use_normals) | (ndot >= cos_min))
        inlier = visible & ok
        reach = d0 <= tau * (1 + DIST_TOL)
        border |= visible & (np.abs(d0 - tau) <= DIST_TOL * tau)
        if use_normals:
            border |= visible & reach & (np.abs(ndot - cos_min) <= DOT_TOL)
        if k > 1:
            border |= visible & reach & (dd[:, 1] - d0 <= TIE_TOL * np.maximum(d0, 1e-12))
    n_in, n_vis = int(inlier.sum()), int(visible.sum())
    rms = float(np.sqrt(np.mean(d0[inlier] ** 2))) if n_in else 0.0
    return dict(inliers=n_in, visible=n_vis, fit=n_in / n_vis if n_vis else 0.0, rms=rms, inlier=inlier, visible_mask=visible,
                borderline=border)
