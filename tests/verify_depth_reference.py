"""Float64 restatement of b200ppf_score_poses_depth (include/b200ppf.h, verification against the depth image).

For a model (N, 6), a scene (M, 6), a pose T (model -> scene, camera at the origin), a depth image D (rows, cols) with
K = fx, fy, ppx, ppy and tau = inlier_dist: model point p moves to p' = R p + t (summed in the device's order, so the bits
agree); it projects to u = floor(fx x'/z' + ppx + 0.5), v = floor(fy y'/z' + ppy + 0.5) and is in view when z' > 0 and
(u, v) lies in the image.  Every in-view point writes z' into the square of half-width min(floor(fx tau / (2 z')), 16) around
its pixel (np.minimum.at); a facing, in-view point is self-occluded when z' > zbuf + tau.  A visible point is unknown where D
has no measurement, occluded when z' > d + tau, a violation when z' < d - tau, and otherwise consistent; the consistent
points take the nearest-neighbour test of tests/verify_reference.py.

score_depth() also returns the borderline points whose outcome rounding may flip: a projection within 1e-9 of a pixel edge,
|z' - d| within 1e-9 max(1, d) of tau, z' within 1e-9 of zbuf + tau, a facing test within 1e-6 of its bound, and the
nearest-neighbour borderline of verify_reference."""
import numpy as np

from verify_reference import DOT_TOL, score

SPLAT_MAX = 16
EDGE_TOL = 1e-9


def move(model, pose):
    """p' and n' (N, 3) as the device sums them: R[r,0] x + R[r,1] y + R[r,2] z + t[r], left to right"""
    m = np.asarray(model, np.float32).astype(np.float64)
    T = np.asarray(pose, np.float64).reshape(4, 4)
    p = np.stack([T[r, 0] * m[:, 0] + T[r, 1] * m[:, 1] + T[r, 2] * m[:, 2] + T[r, 3] for r in range(3)], 1)
    n = np.stack([T[r, 0] * m[:, 3] + T[r, 1] * m[:, 4] + T[r, 2] * m[:, 5] for r in range(3)], 1)
    return p, n


def project(p, K, shape):
    """-> (u, v, in_view, fu, fv) with fu, fv the values floored"""
    fx, fy, ppx, ppy = (float(k) for k in K)
    rows, cols = shape
    z = p[:, 2]
    with np.errstate(divide="ignore", invalid="ignore", over="ignore"):
        fu = fx * p[:, 0] / z + ppx + 0.5
        fv = fy * p[:, 1] / z + ppy + 0.5
    ok = (z > 0) & (fu >= 0) & (fu < cols) & (fv >= 0) & (fv < rows)
    u = np.where(ok, np.floor(np.where(ok, fu, 0)), -1).astype(np.int64)
    v = np.where(ok, np.floor(np.where(ok, fv, 0)), -1).astype(np.int64)
    return u, v, ok, fu, fv


def splat_half(z, fx, tau):
    return np.minimum(np.floor(fx * tau / (2.0 * z)), SPLAT_MAX).astype(np.int64)


def zbuffer(p, u, v, in_view, K, shape, tau):
    """the per-pose z-buffer (rows, cols), inf where no splat reaches"""
    rows, cols = shape
    zb = np.full(rows * cols, np.inf)
    idx = np.flatnonzero(in_view)
    if len(idx) == 0:
        return zb.reshape(shape)
    z = p[idx, 2]
    h = splat_half(z, float(K[0]), tau)
    for hh in np.unique(h):
        sel = h == hh
        for dv in range(-hh, hh + 1):
            for du in range(-hh, hh + 1):
                uu, vv = u[idx[sel]] + du, v[idx[sel]] + dv
                ok = (uu >= 0) & (uu < cols) & (vv >= 0) & (vv < rows)
                np.minimum.at(zb, vv[ok] * cols + uu[ok], z[sel][ok])
    return zb.reshape(shape)


def score_depth(model, scene, pose, depth, K, inlier_dist=0.01, normal_angle=np.radians(30.0)):
    """-> dict(inliers, judged, visible, self_occluded, occluded, violations, unknown, fit, rms, masks..., borderline (N,) bool)"""
    model = np.asarray(model, np.float32).reshape(-1, 6)
    depth = np.asarray(depth, np.float32)
    tau = float(np.float32(inlier_dist))
    p, n = move(model, pose)
    zero = np.all(model[:, 3:6] == 0, axis=1)
    vdot = -(n[:, 0] * p[:, 0] + n[:, 1] * p[:, 1] + n[:, 2] * p[:, 2])
    facing = zero | (vdot > 0)
    u, v, in_view, fu, fv = project(p, K, depth.shape)
    zb = zbuffer(p, u, v, in_view, K, depth.shape, tau)
    z = p[:, 2]
    zpix = np.where(in_view, zb[np.clip(v, 0, None), np.clip(u, 0, None)], np.inf)
    cand = facing & in_view
    self_occ = cand & (z > zpix + tau)
    visible = cand & ~self_occ
    d = np.where(in_view, depth[np.clip(v, 0, None), np.clip(u, 0, None)], 0).astype(np.float64)
    measured = (d > 0) & np.isfinite(d)
    unknown = visible & ~measured
    occluded = visible & measured & (z > d + tau)
    violation = visible & measured & ~occluded & (z < d - tau)
    consistent = visible & measured & ~occluded & ~violation
    judged = visible & measured & ~occluded
    r = score(model[consistent], scene, pose, inlier_dist, normal_angle)
    inlier = np.zeros(len(model), bool)
    inlier[np.flatnonzero(consistent)[r["inlier"]]] = True
    # borderline: rounding may flip the outcome
    border = ~zero & (np.abs(vdot) <= DOT_TOL)
    with np.errstate(invalid="ignore"):
        for f in (fu, fv):
            frac = f - np.floor(f)
            border |= (z > 0) & np.isfinite(f) & ((frac <= EDGE_TOL) | (frac >= 1 - EDGE_TOL))
        border |= cand & np.isfinite(zpix) & (np.abs(z - (zpix + tau)) <= EDGE_TOL)
        border |= visible & measured & (np.abs(np.abs(z - d) - tau) <= EDGE_TOL * np.maximum(1.0, d))
    border[np.flatnonzero(consistent)[r["borderline"]]] = True
    c = dict(inliers=int(inlier.sum()), judged=int(judged.sum()), visible=int(visible.sum()), self_occluded=int(self_occ.sum()),
             occluded=int(occluded.sum()), violations=int(violation.sum()), unknown=int(unknown.sum()))
    c["fit"] = c["inliers"] / c["judged"] if c["judged"] else 0.0
    c["rms"] = r["rms"]
    c.update(inlier=inlier, visible_mask=visible, self_occluded_mask=self_occ, occluded_mask=occluded, violation_mask=violation,
             unknown_mask=unknown, borderline=border)
    return c
