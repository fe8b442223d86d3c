"""A float64 NumPy restatement of ICP::registerModelToScene, step for step as oracle/icp_oracle.cpp states it.

Helper module for the ICP tests (not a conftest).  It exists to look inside ICP: besides the refined pose it returns,
per iteration, the state the device has to reproduce and the decision margins that a last-bit difference could flip.
A comparison of the device with this restatement is only tight where those margins are non-zero.

Arithmetic follows the oracle operation for operation: float32 where the oracle stores float, float64 elsewhere, sums in
the oracle's sequential order (np.cumsum adds left to right), no fused multiply-adds (the device builds with
-fmad=false, the oracle with -ffp-contract=off).  The nearest-neighbour search is brute force, so it is exact by
construction; ties go to the lowest index everywhere, as on both other sides.
"""
from __future__ import annotations

import math
from dataclasses import dataclass, field

import numpy as np

MAD_FACTOR = np.float32(1.48257968)
NN_CHUNK = 256  # model samples per block of the brute-force distance matrix


def _seqsum(v):
    """left-to-right float64 sum, the order of a plain C loop"""
    v = np.asarray(v, np.float64).ravel()
    return float(np.cumsum(v)[-1]) if v.size else 0.0


def mat4_mul(a, b):
    """4 x 4 product with the oracle's summation order (no BLAS)"""
    c = np.zeros((4, 4), np.float64)
    for r in range(4):
        for k in range(4):
            s = 0.0
            for q in range(4):
                s += float(a[r, q]) * float(b[q, k])
            c[r, k] = s
    return c


def transform_cloud(pc, P, with_normals=True):
    """transformPCPose: xyz -> (R p + t) / w, normals -> normalised R n; float32 in, float64 maths, float32 out"""
    pc = np.asarray(pc, np.float32)
    x, y, z = (pc[:, c].astype(np.float64) for c in range(3))
    w = P[3, 0] * x + P[3, 1] * y + P[3, 2] * z + P[3, 3]
    w = np.where(w == 0.0, 1.0, w)
    out = np.empty_like(pc)
    for r in range(3):
        out[:, r] = ((P[r, 0] * x + P[r, 1] * y + P[r, 2] * z + P[r, 3]) / w).astype(np.float32)
    if with_normals:
        nx, ny, nz = (pc[:, 3 + c].astype(np.float64) for c in range(3))
        rn = [P[r, 0] * nx + P[r, 1] * ny + P[r, 2] * nz for r in range(3)]
        ln = np.sqrt(rn[0] * rn[0] + rn[1] * rn[1] + rn[2] * rn[2])
        big = ln > 1e-12
        for r in range(3):
            out[:, 3 + r] = np.where(big, rn[r] / np.where(big, ln, 1.0), rn[r]).astype(np.float32)
    else:
        out = out[:, :3]
    return out


def nearest(q, pts):
    """exact nearest of every query among pts (float32 squared distances summed as (dx*dx + dy*dy) + dz*dz, ties to the
    lowest index) -> (index, d2, gap): gap is the distance from the best d2 to the next larger one (exact ties excluded;
    inf when every sample is at the best distance)"""
    q = np.asarray(q, np.float32)
    pts = np.asarray(pts, np.float32)
    m = q.shape[0]
    idx = np.empty(m, np.int64)
    d2 = np.empty(m, np.float32)
    gap = np.empty(m, np.float64)
    px, py, pz = pts[:, 0][None, :], pts[:, 1][None, :], pts[:, 2][None, :]
    for s in range(0, m, NN_CHUNK):
        e = min(m, s + NN_CHUNK)
        dx = q[s:e, 0][:, None] - px
        dy = q[s:e, 1][:, None] - py
        dz = q[s:e, 2][:, None] - pz
        D = dx * dx + dy * dy + dz * dz
        b = np.argmin(D, axis=1)  # first occurrence: lowest index on ties
        best = D[np.arange(e - s), b]
        second = np.where(D > best[:, None], D, np.float32(np.inf)).min(axis=1)
        idx[s:e] = b
        d2[s:e] = best
        gap[s:e] = second.astype(np.float64) - best.astype(np.float64)
    return idx, d2, gap


def lower_median(v):
    v = np.asarray(v)
    return v[np.argpartition(v, (v.size - 1) // 2)[(v.size - 1) // 2]]


def rejection_threshold(d2, scale):
    """median + scale * 1.48257968 * MAD of the float32 squared distances (lower medians, MAD in double cast to float)"""
    med = np.float32(lower_median(d2))
    t = np.abs(d2.astype(np.float64) - np.float64(med)).astype(np.float32)
    s = MAD_FACTOR * np.float32(lower_median(t))
    return np.float32(np.float32(scale) * s + med), med


JACOBI_ROUNDS = (((0, 5), (1, 4), (2, 3)), ((1, 5), (0, 2), (3, 4)), ((2, 5), (1, 3), (0, 4)),
                 ((3, 5), (2, 4), (0, 1)), ((4, 5), (0, 3), (1, 2)))


def solve6_min_norm(A, b):
    """minimum-norm solve from the Gram matrix by cyclic Jacobi rotations (icp_oracle.cpp solve6_min_norm)
    -> (x or None, smallest |l - cut| / cut over the six eigenvalues)"""
    A = [float(v) for v in np.asarray(A, np.float64).ravel()]
    V = [1.0 if r == c else 0.0 for r in range(6) for c in range(6)]
    for _ in range(30):
        off = diag = 0.0
        for p in range(6):
            diag += abs(A[p * 6 + p])
            for q in range(p + 1, 6):
                off += abs(A[p * 6 + q])
        if not off > 1e-300 or off <= 1e-18 * diag:
            break
        for rnd in JACOBI_ROUNDS:
            cs = []
            for p, q in rnd:
                apq = A[p * 6 + q]
                if apq == 0.0:
                    cs.append((1.0, 0.0))
                    continue
                theta = (A[q * 6 + q] - A[p * 6 + p]) / (2.0 * apq)
                t = (1.0 if theta >= 0.0 else -1.0) / (abs(theta) + math.sqrt(theta * theta + 1.0))
                c = 1.0 / math.sqrt(t * t + 1.0)
                cs.append((c, t * c))
            for (p, q), (c, sn) in zip(rnd, cs):
                for k in range(6):
                    akp, akq = A[k * 6 + p], A[k * 6 + q]
                    A[k * 6 + p] = c * akp - sn * akq
                    A[k * 6 + q] = sn * akp + c * akq
                    vkp, vkq = V[k * 6 + p], V[k * 6 + q]
                    V[k * 6 + p] = c * vkp - sn * vkq
                    V[k * 6 + q] = sn * vkp + c * vkq
            for (p, q), (c, sn) in zip(rnd, cs):
                for k in range(6):
                    apk, aqk = A[p * 6 + k], A[q * 6 + k]
                    A[p * 6 + k] = c * apk - sn * aqk
                    A[q * 6 + k] = sn * apk + c * aqk
    lmax = 0.0
    for k in range(6):
        lmax = max(lmax, A[k * 6 + k])  # fmax: a NaN diagonal entry is skipped
    if not lmax > 0.0:
        return None, math.inf
    cut = 1e-12 * lmax
    x = [0.0] * 6
    margin = math.inf
    for k in range(6):
        lam = A[k * 6 + k]
        margin = min(margin, abs(lam - cut) / cut)
        if not lam > cut:
            continue
        proj = 0.0
        for r in range(6):
            proj += V[r * 6 + k] * float(b[r])
        proj /= lam
        for r in range(6):
            x[r] += V[r * 6 + k] * proj
    if not all(math.isfinite(v) for v in x):
        return None, margin
    return np.array(x), margin


def solve6(A, b):
    """elimination with partial pivoting while every pivot exceeds 1e-9 of the largest diagonal entry, else the
    minimum-norm form (icp_oracle.cpp solve6) -> (x or None, branch, pivot margin, eigenvalue margin); the pivot margin
    is the smallest | |pivot| - floor | / floor over the pivots taken, the eigenvalue margin that of solve6_min_norm
    (inf on the elimination branch)"""
    A = np.asarray(A, np.float64).reshape(6, 6)
    b = np.asarray(b, np.float64).reshape(6)
    E = [float(v) for v in A.ravel()]
    g = [float(v) for v in b]
    dmax = 0.0
    for k in range(6):
        dmax = max(dmax, abs(E[k * 6 + k]))
    floor_pivot = 1e-9 * dmax
    perm = list(range(6))
    full_rank = dmax > 0.0
    pivot_margin = math.inf
    c = 0
    while c < 6 and full_rank:
        piv = c
        for r in range(c + 1, 6):
            if abs(E[perm[r] * 6 + c]) > abs(E[perm[piv] * 6 + c]):
                piv = r
        perm[c], perm[piv] = perm[piv], perm[c]
        d = E[perm[c] * 6 + c]
        pivot_margin = min(pivot_margin, abs(abs(d) - floor_pivot) / floor_pivot)
        if not abs(d) > floor_pivot:
            full_rank = False
            break
        for r in range(c + 1, 6):
            f = E[perm[r] * 6 + c] / d
            for k in range(c, 6):
                E[perm[r] * 6 + k] -= f * E[perm[c] * 6 + k]
            g[perm[r]] -= f * g[perm[c]]
        c += 1
    if not full_rank:
        x, eig_margin = solve6_min_norm(A, b)
        return x, "min_norm", pivot_margin, eig_margin
    x = [0.0] * 6
    for c in range(5, -1, -1):
        s = g[perm[c]]
        for k in range(c + 1, 6):
            s -= E[perm[c] * 6 + k] * x[k]
        x[c] = s / E[perm[c] * 6 + c]
    if not all(math.isfinite(v) for v in x):
        return None, "elimination", pivot_margin, math.inf
    return np.array(x), "elimination", pivot_margin, math.inf


def pose_from_euler(rpy, t):
    """[Rx(roll) Ry(pitch) Rz(yaw) | t] with the oracle's product order"""
    cx, sx = math.cos(rpy[0]), math.sin(rpy[0])
    cy, sy = math.cos(rpy[1]), math.sin(rpy[1])
    cz, sz = math.cos(rpy[2]), math.sin(rpy[2])
    Rx = (1.0, 0.0, 0.0, 0.0, cx, -sx, 0.0, sx, cx)
    Ry = (cy, 0.0, sy, 0.0, 1.0, 0.0, -sy, 0.0, cy)
    Rz = (cz, -sz, 0.0, sz, cz, 0.0, 0.0, 0.0, 1.0)
    T = [Ry[r * 3] * Rz[c] + Ry[r * 3 + 1] * Rz[3 + c] + Ry[r * 3 + 2] * Rz[6 + c] for r in range(3) for c in range(3)]
    R = [Rx[r * 3] * T[c] + Rx[r * 3 + 1] * T[3 + c] + Rx[r * 3 + 2] * T[6 + c] for r in range(3) for c in range(3)]
    P = np.eye(4)
    for r in range(3):
        for c in range(3):
            P[r, c] = R[r * 3 + c]
        P[r, 3] = float(t[r])
    return P


@dataclass
class Iteration:
    """what one iteration decided, and how far each decision was from flipping"""
    level: int
    samples: int          # model samples m of the level
    matches: int          # surviving pairs in the normal equations
    threshold: float      # rejection threshold (inf when rejection_scale <= 0)
    branch: str           # "elimination" or "min_norm"
    nn_gap: float         # smallest gap between best and second-best d2 of any model sample (exact ties excluded)
    thr_gap: float        # smallest |d2 - threshold|
    winner_gap: float     # smallest gap between the winning and the next d2 on one scene sample (exact ties excluded)
    pivot_margin: float   # smallest | |pivot| - 1e-9 dmax | / (1e-9 dmax)
    eig_margin: float     # smallest |l - 1e-12 lmax| / (1e-12 lmax) (minimum-norm branch only)
    fperc_gap: float      # |fperc - (1 +- tol)|, the nearer of the two
    fval: float


@dataclass
class Result:
    pose: np.ndarray
    residual: float
    iterations: int
    trace: list = field(default_factory=list)   # Iteration records, in order
    levels: list = field(default_factory=list)  # (level, m, md, step, max_it) of every level that ran

    def margins(self):
        """the smallest of every decision margin over all iterations"""
        keys = ("nn_gap", "thr_gap", "winner_gap", "pivot_margin", "eig_margin", "fperc_gap")
        return {k: min((getattr(t, k) for t in self.trace), default=math.inf) for k in keys}


def _register_single(src, dst, max_iterations, tolerance, rejection_scale, num_levels):
    n, nd = src.shape[0], dst.shape[0]
    src, dst = src.copy(), dst.copy()
    ms = [_seqsum(src[:, c]) for c in range(3)]
    md = [_seqsum(dst[:, c]) for c in range(3)]
    mean = [0.5 * (ms[c] / n + md[c] / nd) for c in range(3)]

    def centre(pc):
        for c in range(3):
            pc[:, c] = (pc[:, c].astype(np.float64) - mean[c]).astype(np.float32)
        x, y, z = (pc[:, c].astype(np.float64) for c in range(3))
        return _seqsum(np.sqrt(x * x + y * y + z * z))

    dist_src, dist_dst = centre(src), centre(dst)
    scale = n / ((dist_src + dist_dst) * 0.5)
    src[:, :3] = (src[:, :3].astype(np.float64) * scale).astype(np.float32)
    dst[:, :3] = (dst[:, :3].astype(np.float64) * scale).astype(np.float32)

    pose = np.eye(4)
    residual = 0.0
    trace, levels = [], []
    iterations = 0
    tol32 = float(np.float32(tolerance))
    for level in range(num_levels - 1, -1, -1):
        div = 2.0 ** level
        num_samples = int(np.rint(n / div))
        tol_p = tol32 * (level + 1) * (level + 1)
        max_it = int(np.rint(max_iterations / (level + 1)))
        if num_samples < 1:
            continue
        step = max(1, int(np.rint(n / num_samples)))
        src_t = transform_cloud(src, pose)[::step]
        dst_s = dst[::step]
        m, mds = src_t.shape[0], dst_s.shape[0]
        levels.append((level, m, mds, step, max_it))
        fval_old, fval_perc, fval_min = 9999999999.0, 0.0, 9999999999.0
        moved = src_t[:, :3].copy()
        pose_x = np.eye(4)
        it = 0
        while not (fval_perc < 1.0 + tol_p and fval_perc > 1.0 - tol_p) and it < max_it:
            nn, d2, gap = nearest(moved, dst_s)
            if rejection_scale > 0.0:
                thr, _ = rejection_threshold(d2, rejection_scale)
                keep = d2 < thr
                thr_gap = float(np.min(np.abs(d2.astype(np.float64) - np.float64(thr))))
            else:
                thr = np.float32(np.inf)
                keep = np.ones(m, bool)
                thr_gap = math.inf
            # of several model samples on one scene sample the closest survives (lowest index on ties)
            ki = np.flatnonzero(keep)
            order = ki[np.lexsort((ki, d2[ki], nn[ki]))]
            first = np.ones(order.size, bool)
            first[1:] = nn[order][1:] != nn[order][:-1]
            win_i = order[first]
            win_j = nn[win_i]
            # the next larger d2 on the same scene sample, for the winner's margin
            winner_gap = math.inf
            if order.size:
                grp = np.cumsum(first) - 1
                best = d2[win_i][grp]
                later = d2[order] > best
                if later.any():
                    nxt = np.full(win_i.size, np.inf)
                    np.minimum.at(nxt, grp[later], d2[order][later].astype(np.float64))
                    winner_gap = float(np.min(nxt - d2[win_i].astype(np.float64)))
            srt = np.argsort(win_j, kind="stable")  # the oracle walks the scene samples in order
            win_i, win_j = win_i[srt], win_j[srt]
            matches = win_i.size
            if matches == 0:
                break
            s = src_t[win_i].astype(np.float64)
            d = dst_s[win_j].astype(np.float64)
            sp, dp, nr = s[:, :3], d[:, :3], d[:, 3:6]
            row = np.stack([sp[:, 1] * nr[:, 2] - sp[:, 2] * nr[:, 1], sp[:, 2] * nr[:, 0] - sp[:, 0] * nr[:, 2],
                            sp[:, 0] * nr[:, 1] - sp[:, 1] * nr[:, 0], nr[:, 0], nr[:, 1], nr[:, 2]], axis=1)
            rhs = (dp[:, 0] - sp[:, 0]) * nr[:, 0] + (dp[:, 1] - sp[:, 1]) * nr[:, 1] + (dp[:, 2] - sp[:, 2]) * nr[:, 2]
            A = np.array([[_seqsum(row[:, r] * row[:, c]) for c in range(6)] for r in range(6)])
            bb = np.array([_seqsum(row[:, r] * rhs) for r in range(6)])
            e = s - d
            err2 = _seqsum(e * e)  # row by row, six columns each: the oracle's order
            x, branch, pivot_margin, eig_margin = solve6(A, bb)
            if x is None:
                break
            pose_x = pose_from_euler(x[:3], x[3:])
            moved = transform_cloud(src_t, pose_x, with_normals=False)
            fval = math.sqrt(err2) / m
            fval_perc = fval / fval_old
            fval_old = fval
            fval_min = min(fval_min, fval)
            it += 1
            iterations += 1
            trace.append(Iteration(level, m, matches, float(thr), branch, float(np.min(gap)), thr_gap, winner_gap,
                                   pivot_margin, eig_margin,
                                   min(abs(fval_perc - (1.0 + tol_p)), abs(fval_perc - (1.0 - tol_p))), fval))
        pose = mat4_mul(pose_x, pose)
        residual = fval_min
    t = [pose[r, 3] / scale + mean[r] - (pose[r, 0] * mean[0] + pose[r, 1] * mean[1] + pose[r, 2] * mean[2])
         for r in range(3)]
    for r in range(3):
        pose[r, 3] = t[r]
    return pose, residual, iterations, trace, levels


def register(model, scene, pose, max_iterations=100, tolerance=0.005, rejection_scale=2.5, num_levels=8):
    """ICP::registerModelToScene for one start pose (model -> scene, 4 x 4): -> Result with the refined pose
    (Pose3D::appendPose: delta * start), the residual, the iteration count and the per-iteration trace"""
    model = np.ascontiguousarray(model, np.float32).reshape(-1, 6)
    scene = np.ascontiguousarray(scene, np.float32).reshape(-1, 6)
    start = np.asarray(pose, np.float64).reshape(4, 4)
    moved = transform_cloud(model, start)
    delta, residual, iterations, trace, levels = _register_single(moved, scene, max_iterations, np.float32(tolerance),
                                                                   float(np.float32(rejection_scale)), num_levels)
    return Result(mat4_mul(delta, start), residual, iterations, trace, levels)
