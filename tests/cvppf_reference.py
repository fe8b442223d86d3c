"""A float64 NumPy restatement of cv::ppf_match_3d::PPF3DDetector (trainModel, match, match_S2B, clusterPoses), written
from upstream's definitions (ppf_match_3d.cpp, ppf_helpers.cpp, c_utils.hpp, hash_murmur86.hpp, pose_3d.cpp).

Helper module for the OpenCV engine's tests (not a conftest).  It calls neither oracle/cvppf_oracle.cpp nor the device
engine (csrc/k7_cvppf.cu); both are compared with it.  Besides the results it lists every decision a last-bit
difference could flip, with its distance to the nearest edge:
  - the three angle keys and the distance key of every model pair and every scene pair ((int) truncation of f / step);
  - the alpha index of every vote ((int)(N (alpha + 2 pi) / 4 pi));
  - the float(alpha) rounding of every alpha_m entry;
  - the branches of Pose3D::updatePose (angle from the trace, the quaternion's branch-on-largest form);
  - the two threshold comparisons of clusterPoses for every leader a pose is tested against.
The device's sin / cos / acos / atan2 may differ from glibc's (and NumPy's) in the last ulp, so a comparison is only
bit-exact where no decision sits on an edge.  A decision is safe if its quantity is exactly 0 or lies more than
SAFE = 1e-9 of a bin width from an edge (a threshold comparison: 1e-9 of the threshold).  For float(alpha) the bin is
one float32 ulp, and 1e-9 of it is half a double ulp (2^-29 of a float ulp), so there the bar is FLOAT_SAFE = 2^-25
of a float ulp: 16 double ulps of the atan2 result.

Arithmetic follows upstream operation for operation: float32 where upstream stores float (the sampling cell index, the
diameter, the distance step, alpha_m), float64 elsewhere, dot products and sums left to right, no fused multiply-adds.
"""
from __future__ import annotations

import math
from dataclasses import dataclass, field

import numpy as np

CV_EPS = 1.192092896e-07  # EPS of c_utils.hpp
PI = math.pi
SAFE = 1e-9
FLOAT_SAFE = 2.0 ** -25
TABLE_MAX_POINTS = 46340  # largest m with m^2 <= 2^31: the device table's 32-bit limit


# ---- decision margins -------------------------------------------------------------------------------------------------
@dataclass
class Margins:
    """per kind of decision: how many were taken, how many are unsafe, the smallest margin (in bin widths)"""
    stats: dict = field(default_factory=dict)

    def add(self, name, margin, bar=SAFE):
        margin = np.asarray(margin, np.float64).ravel()
        if margin.size == 0:
            return
        n, bad, low = self.stats.get(name, (0, 0, np.inf))
        self.stats[name] = (n + margin.size, bad + int(np.count_nonzero(~(margin > bar))), min(low, float(margin.min())))

    def unsafe(self):
        return sum(bad for _, bad, _ in self.stats.values())

    def report(self):
        return {k: {"decisions": n, "unsafe": bad, "min_margin": low} for k, (n, bad, low) in self.stats.items()}


def trunc_margin(x):
    """distance, in bins, of x from the nearest edge of (int)x: the integers other than 0 (truncation maps (-1, 1) to 0)"""
    x = np.asarray(x, np.float64)
    e = np.rint(x)
    e = np.where(e == 0, np.where(x < 0, -1.0, 1.0), e)
    return np.abs(x - e)


def float_round_margin(a):
    """distance of a double from the midpoint between the two float32 values around it, in float32 ulps (0.5 when the
    double is a float32 value)"""
    a = np.asarray(a, np.float64)
    f = a.astype(np.float32)
    g = np.where(a > f, np.nextafter(f, np.float32(np.inf)), np.nextafter(f, np.float32(-np.inf)))
    width = np.abs(g.astype(np.float64) - f.astype(np.float64))
    mid = (f.astype(np.float64) + g.astype(np.float64)) / 2
    return np.where(a == f, 0.5, np.abs(a - mid) / width)


# ---- samplePCByQuantization -------------------------------------------------------------------------------------------
def bbox(pc):
    """computeBboxStd: per axis (min, max) of the float32 coordinates"""
    xyz = np.asarray(pc, np.float32)[:, :3]
    return xyz.min(axis=0), xyz.max(axis=0)


def sample_cells(pc, sample_step):
    """(cell index of every point, ns): (int)((float)ns * (x - lo) / extent) per axis in float32, combined with upstream's
    stride ns although a coordinate on the upper bound lands in cell ns (such points share a neighbouring cell's list)"""
    pc = np.asarray(pc, np.float32)
    ns = int(1.0 / float(np.float32(sample_step)))
    lo, hi = bbox(pc)
    ext = hi - lo
    c = ((np.float32(ns) * (pc[:, :3] - lo)) / ext).astype(np.int64)  # float32 product and quotient, truncation
    return c[:, 0] * ns * ns + c[:, 1] * ns + c[:, 2], ns


def sample(pc, sample_step):
    """samplePCByQuantization (weightByCenter = 0) over the cloud's own bounding box: the points of a cell averaged in
    double in input order, the normal renormalised (left at 0 when its norm is <= EPS); cells in ascending index order"""
    pc = np.asarray(pc, np.float32)
    index, _ = sample_cells(pc, sample_step)
    order = np.argsort(index, kind="stable")
    si = index[order]
    starts = np.flatnonzero(np.r_[True, si[1:] != si[:-1]])
    counts = np.diff(np.r_[starts, si.size])
    a = np.zeros((starts.size, 6), np.float64)
    for k in range(int(counts.max())):  # sequential sums: the k-th member of every cell that has one
        sel = counts > k
        a[sel] += pc[order[starts[sel] + k], :6].astype(np.float64)
    a /= counts[:, None].astype(np.float64)
    nn = np.sqrt(a[:, 3] * a[:, 3] + a[:, 4] * a[:, 4] + a[:, 5] * a[:, 5])
    out = np.zeros((starts.size, 6), np.float32)
    out[:, :3] = a[:, :3].astype(np.float32)
    big = nn > CV_EPS
    out[big, 3:] = (a[big, 3:] / nn[big, None]).astype(np.float32)
    return out


# ---- pair features, hash, frames ---------------------------------------------------------------------------------------
def _cross_norm(ax, ay, az, bx, by, bz):
    cx = ay * bz - az * by
    cy = az * bx - ax * bz
    cz = ax * by - ay * bx
    return np.sqrt(cx * cx + cy * cy + cz * cz)


def _angle3(ax, ay, az, bx, by, bz):
    """TAngle3Normalized: atan2(|a x b|, a . b)"""
    cx = ay * bz - az * by
    cy = az * bx - ax * bz
    cz = ax * by - ay * bx
    return np.arctan2(np.sqrt(cx * cx + cy * cy + cz * cz), ax * bx + ay * by + az * bz)


def features(p1, n1, p2, n2):
    """computePPFFeatures on float64 (..., 3) arrays (broadcast) -> (f (..., 4), exact (..., 3)): f0..f2 stay 0 when
    |d| <= EPS, f3 = |d|.  exact marks the angles whose atan2 has y = 0: atan2(+-0, x) is +-0 or +-pi exactly (C99
    Annex F, which CUDA's atan2 follows too), so their keys are the same on every side even on a bin edge (an
    antiparallel pair gives pi; a zero normal gives atan2(0, -0) = pi when every component of d is negative)"""
    dx, dy, dz = (p2[..., k] - p1[..., k] for k in range(3))
    f3 = np.sqrt(dx * dx + dy * dy + dz * dz)
    small = f3 <= CV_EPS
    inv = 1.0 / np.where(small, 1.0, f3)
    ux, uy, uz = dx * inv, dy * inv, dz * inv
    n1x, n1y, n1z = (n1[..., k] for k in range(3))
    n2x, n2y, n2z = (n2[..., k] for k in range(3))
    f = np.empty(np.broadcast(f3, n1x, n2x).shape + (4,), np.float64)
    f[..., 0] = np.where(small, 0.0, _angle3(n1x, n1y, n1z, ux, uy, uz))
    f[..., 1] = np.where(small, 0.0, _angle3(n2x, n2y, n2z, ux, uy, uz))
    f[..., 2] = np.where(small, 0.0, _angle3(n1x, n1y, n1z, n2x, n2y, n2z))
    f[..., 3] = f3
    exact = np.stack([small | (_cross_norm(n1x, n1y, n1z, ux, uy, uz) == 0), small | (_cross_norm(n2x, n2y, n2z, ux, uy, uz) == 0),
                      small | (_cross_norm(n1x, n1y, n1z, n2x, n2y, n2z) == 0)], axis=-1)
    return f, exact


def quantise(f, exact, angle_step, distance_step, margins=None, label=""):
    """hashPPF's key: the four features truncated to int32 by their steps; the four truncations go to margins (an exact
    angle's at an infinite margin)"""
    q = np.empty(f.shape, np.float64)
    q[..., :3] = f[..., :3] / angle_step
    q[..., 3] = f[..., 3] / distance_step
    if margins is not None:
        margins.add(label + "angle key", np.where(exact, np.inf, trunc_margin(q[..., :3])))
        margins.add(label + "distance key", trunc_margin(q[..., 3]))
    return np.trunc(q).astype(np.int32)


def _rotl(x, r):
    return (x << np.uint32(r)) | (x >> np.uint32(32 - r))


def murmur3_x86_32(words, seed=42):
    """MurmurHash3_x86_32 of rows of 32-bit words (..., n) (little-endian bytes of the row), vectorised over the rows"""
    w = np.ascontiguousarray(words).view(np.uint32)
    with np.errstate(over="ignore"):
        h = np.full(w.shape[:-1], seed, np.uint32)
        for i in range(w.shape[-1]):
            k = w[..., i] * np.uint32(0xCC9E2D51)
            k = _rotl(k, 15) * np.uint32(0x1B873593)
            h = _rotl(h ^ k, 13) * np.uint32(5) + np.uint32(0xE6546B64)
        h = h ^ np.uint32(4 * w.shape[-1])
        h = h ^ (h >> np.uint32(16))
        h = h * np.uint32(0x85EBCA6B)
        h = h ^ (h >> np.uint32(13))
        h = h * np.uint32(0xC2B2AE35)
        h = h ^ (h >> np.uint32(16))
    return h


def transform_rt(p, n):
    """computeTransformRT for rows (K, 3): the rotation aaToR(n x e_x, acos(n_x)) taking n onto the x axis, t = -R p"""
    p, n = np.asarray(p, np.float64), np.asarray(n, np.float64)
    angle = np.arccos(n[:, 0])
    ax = np.zeros(len(n))
    ay, az = n[:, 2].copy(), -n[:, 1]
    special = (n[:, 1] == 0) & (n[:, 2] == 0)
    nn = np.sqrt(ax * ax + ay * ay + az * az)
    scale = ~special & (nn > CV_EPS)
    ay = np.where(special, 1.0, np.where(scale, ay / np.where(scale, nn, 1.0), ay))
    az = np.where(special, 0.0, np.where(scale, az / np.where(scale, nn, 1.0), az))
    a = (ax, ay, az)
    s, c = np.sin(angle), np.cos(angle)
    c1 = 1.0 - c
    R = np.empty((len(n), 3, 3), np.float64)
    for i in range(3):
        for j in range(3):
            v = c if i == j else np.zeros(len(n))
            if i != j:
                v = v + ((-1.0 if (i + 1) % 3 == j else 1.0) * s) * a[3 - i - j]
            R[:, i, j] = v + (c1 * a[i]) * a[j]
    t = -mat_vec(R, p)
    return R, t


def mat_vec(R, v):
    """rows of R (K, 3, 3) times v (K, 3) or (3,), each entry summed left to right"""
    v = np.broadcast_to(v, R.shape[:-2] + (3,)) if v.ndim == 1 else v
    return np.stack([R[..., r, 0] * v[..., 0] + R[..., r, 1] * v[..., 1] + R[..., r, 2] * v[..., 2] for r in range(3)], axis=-1)


def planar_alpha(R, t, p2):
    """computeAlpha: planar angle of p2 in the frame (R, t) -> (alpha, is_nan); R (3, 3), t (3,), p2 (K, 3)"""
    rp = np.stack([R[r, 0] * p2[:, 0] + R[r, 1] * p2[:, 1] + R[r, 2] * p2[:, 2] for r in range(3)], axis=-1)
    my, mz = t[1] + rp[:, 1], t[2] + rp[:, 2]
    a = np.arctan2(-mz, my)
    is_nan = np.isnan(a)
    a = np.where(np.sin(a) * mz < 0.0, -a, a)
    return np.where(is_nan, 0.0, -a), is_nan


def alpha_index(alpha, num_angles):
    """(int)(numAngles * (alpha + 2 pi) / (4 pi)) as double arithmetic, and the quantity before the truncation"""
    x = num_angles * (alpha + 2 * PI) / (4 * PI)
    return np.trunc(x).astype(np.int64), x


# ---- trainModel --------------------------------------------------------------------------------------------------------
@dataclass
class Trained:
    model: np.ndarray          # (m, 6) sampled model
    angle_step: float
    distance_step: float       # a float32 value
    num_angles: int            # floor(2 pi / angle_step): the accumulator's columns
    table_size: int
    offsets: np.ndarray        # (table_size + 1,) uint32: CSR over the buckets h & (size - 1)
    nodes: np.ndarray          # ppfInd = i * m + j, ascending inside a bucket
    alpha_m: np.ndarray        # (m * m,) float32, 0 on the diagonal
    margins: Margins
    position_threshold: float
    rotation_threshold: float

    @property
    def m(self):
        return self.model.shape[0]


def steps(num_angles_arg):
    """angle_step = (360 / numAngles) * pi / 180 and the columns floor(2 pi / angle_step) it gives"""
    angle_step = (360.0 / num_angles_arg) * PI / 180.0
    return angle_step, int(math.floor(2 * PI / angle_step))


def train(model_cloud, sampling_step=0.05, num_angles_arg=30, chunk=128):
    """PPF3DDetector(sampling_step, ., num_angles_arg).trainModel(model_cloud); the sampled model must have 2 ..
    TABLE_MAX_POINTS points"""
    pc = np.asarray(model_cloud, np.float32)
    lo, hi = bbox(pc)
    d = hi - lo
    diameter = np.sqrt(d[0] * d[0] + d[1] * d[1] + d[2] * d[2])  # float32
    distance_step = float(np.float32(float(diameter) * sampling_step))
    model = sample(pc, np.float32(sampling_step))
    m = model.shape[0]
    assert 2 <= m <= TABLE_MAX_POINTS, m
    angle_step, num_angles = steps(num_angles_arg)
    size = 16
    while size < m * m:
        size <<= 1
    margins = Margins()
    P, N = model[:, :3].astype(np.float64), model[:, 3:].astype(np.float64)
    R, t = transform_rt(P, N)
    bucket = np.empty(m * m, np.int64)
    alpha_m = np.zeros(m * m, np.float32)
    for i0 in range(0, m, chunk):
        i1 = min(m, i0 + chunk)
        f, exact = features(P[i0:i1, None, :], N[i0:i1, None, :], P[None, :, :], N[None, :, :])
        off_diag = np.ones((i1 - i0, m), bool)
        off_diag[np.arange(i1 - i0), np.arange(i0, i1)] = False
        key = quantise(f[off_diag], exact[off_diag], angle_step, distance_step, margins, "model ")
        b = np.full((i1 - i0, m), -1, np.int64)
        b[off_diag] = murmur3_x86_32(key) & np.uint32(size - 1)
        bucket[i0 * m:i1 * m] = b.ravel()
        for i in range(i0, i1):
            a, _ = planar_alpha(R[i], t[i], P)
            a[i] = 0.0
            alpha_m[i * m:(i + 1) * m] = a.astype(np.float32)
            margins.add("float(alpha)", float_round_margin(np.delete(a, i)), FLOAT_SAFE)
    valid = np.flatnonzero(bucket >= 0)
    nodes = valid[np.argsort(bucket[valid], kind="stable")].astype(np.uint32)  # ascending ppfInd inside a bucket
    offsets = np.searchsorted(bucket[nodes], np.arange(size + 1), side="left").astype(np.uint32)
    return Trained(model, angle_step, distance_step, num_angles, size, offsets, nodes, alpha_m, margins,
                   position_threshold=sampling_step, rotation_threshold=(360.0 / num_angles_arg) / 180.0 * PI)


# ---- match / match_S2B -------------------------------------------------------------------------------------------------
POSE_FIELDS = ("pose", "alpha", "angle", "t", "q", "model_index", "num_votes", "alpha_index", "reference_index")


@dataclass
class Match:
    scene: np.ndarray        # sampled scene (the reference points are every step-th row)
    second: np.ndarray       # the points a reference is paired with: the sampled scene, or the sampled edge cloud
    step: int
    raw: dict                # per reference: POSE_FIELDS arrays
    clusters: list           # dicts: pose, angle, t, q, num_votes, leader (reference), members
    accumulators: dict       # reference -> (m, num_angles) uint32 of the references asked for
    margins: Margins
    overflow: dict           # votes whose alpha index is numAngles: on a row before the last / on the last (dropped)
    overflow_refs: list      # the references that cast such votes
    ties: int                # references whose maximum occurs more than once

    @property
    def refs(self):
        return len(self.raw["num_votes"])


def vote_one(tr: Trained, p1, n1, second, skip, margins=None):
    """the accumulator of one reference point (p1, n1) against the points `second` (row `skip` left out: match() pairs
    a reference with every other sampled point) -> (acc (m, N) uint32, votes with index N before the last row, on it)"""
    m, N = tr.m, tr.num_angles
    keep = np.ones(len(second), bool)
    if skip is not None:
        keep[skip] = False
    p2 = second[keep, :3].astype(np.float64)
    n2 = second[keep, 3:].astype(np.float64)
    f, exact = features(p1[None, :], n1[None, :], p2, n2)
    key = quantise(f, exact, tr.angle_step, tr.distance_step, margins, "scene ")
    h = (murmur3_x86_32(key) & np.uint32(tr.table_size - 1)).astype(np.int64)
    R, t = transform_rt(p1[None, :], n1[None, :])
    alpha_s, is_nan = planar_alpha(R[0], t[0], p2)
    b, e = tr.offsets[h].astype(np.int64), tr.offsets[h + 1].astype(np.int64)
    e = np.where(is_nan, b, e)
    lens = e - b
    pair = np.repeat(np.arange(len(h)), lens)
    pos = np.repeat(b - np.r_[0, np.cumsum(lens)[:-1]], lens) + np.arange(int(lens.sum()))
    node = tr.nodes[pos].astype(np.int64)
    alpha = tr.alpha_m[node].astype(np.float64) - alpha_s[pair]
    idx, x = alpha_index(alpha, N)
    if margins is not None:
        margins.add("alpha index", np.where(alpha == 0.0, np.inf, trunc_margin(x)))
    row = node // m
    cell = row * N + idx
    ok = cell < m * N  # alpha index N on the last row is dropped, as upstream's bound check does
    acc = np.bincount(cell[ok], minlength=m * N).astype(np.uint32).reshape(m, N)
    at_n = idx == N
    return acc, int(np.count_nonzero(at_n & (row < m - 1))), int(np.count_nonzero(at_n & (row == m - 1)))


def _mul44(a, b):
    """4 x 4 products over the leading axis, each entry summed left to right from 0"""
    c = np.zeros(a.shape, np.float64)
    for r in range(4):
        for k in range(4):
            s = np.zeros(a.shape[0])
            for q in range(4):
                s = s + a[:, r, q] * b[:, q, k]
            c[:, r, k] = s
    return c


def _rt_to_pose(R, t):
    T = np.zeros((R.shape[0], 4, 4))
    T[:, :3, :3] = R
    T[:, :3, 3] = t
    T[:, 3, 3] = 1.0
    return T


def update_pose(P, margins=None):
    """Pose3D::updatePose(Matx44d): angle from the trace (0 / pi within EPS of 3 / -1), t, q (w x y z) by the
    branch-on-largest form; the branch decisions go to margins"""
    r = P[:, :3, :3]
    trace = r[:, 0, 0] + r[:, 1, 1] + r[:, 2, 2]
    with np.errstate(invalid="ignore"):  # the arccos of the ends is computed and not taken
        angle = np.where(np.abs(trace - 3) <= CV_EPS, 0.0,
                         np.where(np.abs(trace + 1) <= CV_EPS, PI, np.arccos((trace - 1) / 2)))
    q = np.empty((P.shape[0], 4))
    r00, r01, r02, r10, r11, r12, r20, r21, r22 = (r[:, i, j] for i in range(3) for j in range(3))
    b0 = trace > 0.0
    b1 = ~b0 & (r00 > r11) & (r00 > r22)
    b2 = ~b0 & ~b1 & (r11 > r22)
    b3 = ~b0 & ~b1 & ~b2
    with np.errstate(invalid="ignore", divide="ignore"):
        s = np.sqrt(trace + 1.0) * 2.0
        qa = np.stack([0.25 * s, (r21 - r12) / s, (r02 - r20) / s, (r10 - r01) / s], 1)
        s = np.sqrt(1.0 + r00 - r11 - r22) * 2.0
        qb = np.stack([(r21 - r12) / s, 0.25 * s, (r01 + r10) / s, (r02 + r20) / s], 1)
        s = np.sqrt(1.0 + r11 - r00 - r22) * 2.0
        qc = np.stack([(r02 - r20) / s, (r01 + r10) / s, 0.25 * s, (r12 + r21) / s], 1)
        s = np.sqrt(1.0 + r22 - r00 - r11) * 2.0
        qd = np.stack([(r10 - r01) / s, (r02 + r20) / s, (r12 + r21) / s, 0.25 * s], 1)
    for sel, qq in ((b0, qa), (b1, qb), (b2, qc), (b3, qd)):
        q[sel] = qq[sel]
    if margins is not None:
        margins.add("pose trace", np.minimum(np.abs(np.abs(trace - 3) - CV_EPS), np.abs(np.abs(trace + 1) - CV_EPS)))
        m = np.abs(trace)  # every comparison the branch chain evaluates, a conjunction's both sides included
        m = np.where(b0, m, np.minimum(m, np.minimum(np.abs(r00 - r11), np.abs(r00 - r22))))
        m = np.where(b0 | b1, m, np.minimum(m, np.abs(r11 - r22)))
        margins.add("quaternion branch", m)
    return angle, P[:, :3, 3].copy(), q


def peak_poses(tr: Trained, scene_refs, model_index, alpha_idx, margins=None):
    """the pose Tsg^-1 Rx(alpha) Tmg of every reference's peak, then updatePose"""
    N = tr.num_angles
    Rs, ts = transform_rt(scene_refs[:, :3], scene_refs[:, 3:])
    RInv = np.transpose(Rs, (0, 2, 1))
    rt = mat_vec(RInv, ts)
    TsgInv = _rt_to_pose(RInv, -rt)
    mp = tr.model[model_index]
    Rm, tm = transform_rt(mp[:, :3], mp[:, 3:])
    Tmg = _rt_to_pose(Rm, tm)
    alpha = (alpha_idx.astype(np.float64) * (4 * PI)) / N - 2 * PI
    c, s = np.cos(alpha), np.sin(alpha)
    Rx = np.zeros((len(alpha), 3, 3))
    Rx[:, 0, 0] = 1
    Rx[:, 1, 1], Rx[:, 1, 2], Rx[:, 2, 1], Rx[:, 2, 2] = c, -s, s, c
    P = _mul44(TsgInv, _mul44(_rt_to_pose(Rx, np.zeros((len(alpha), 3))), Tmg))
    angle, t, q = update_pose(P, margins)
    return P, alpha, angle, t, q


def cluster_poses(raw, position_threshold, rotation_threshold, margins=None):
    """clusterPoses: poses sorted by votes (stable: ties in reference order), each joins the first cluster whose FIRST
    pose matches (|angle difference| < rotation threshold and |t difference| < position threshold), clusters sorted by
    vote sum (stable), quaternions and translations averaged in joining order, the quaternion normalised"""
    votes = raw["num_votes"].astype(np.int64)
    order = np.argsort(-votes, kind="stable")
    leaders, members = [], []
    lt = np.zeros((len(order), 3))
    la = np.zeros(len(order))

    def crossing(qty, thr):
        if thr == 0:
            return np.full(qty.shape, np.inf)  # x < 0 never holds for a distance / an absolute value
        return np.abs(qty - thr) / abs(thr)

    for k in order:
        n = len(leaders)
        joined = None
        if n:
            dx, dy, dz = (lt[:n, e] - raw["t"][k, e] for e in range(3))
            dn = np.sqrt(dx * dx + dy * dy + dz * dz)
            phi = np.abs(raw["angle"][k] - la[:n])
            ok_r, ok_p = phi < rotation_threshold, dn < position_threshold
            hit = np.flatnonzero(ok_r & ok_p)
            last = hit[0] if hit.size else n - 1
            if margins is not None:
                # a test is settled if one condition is false with a margin, or both are true with margins
                mr, mp = crossing(phi[:last + 1], rotation_threshold), crossing(dn[:last + 1], position_threshold)
                sure_r, sure_p = mr > SAFE, mp > SAFE
                a, b = ok_r[:last + 1], ok_p[:last + 1]
                settled = (~a & sure_r) | (~b & sure_p) | (a & b & sure_r & sure_p)
                margins.add("cluster threshold", np.where(settled, np.inf, np.minimum(mr, mp)))
            if hit.size:
                joined = int(hit[0])
        if joined is None:
            lt[n], la[n] = raw["t"][k], raw["angle"][k]
            leaders.append(int(k))
            members.append([int(k)])
        else:
            members[joined].append(int(k))
    sums = np.array([int(votes[mm].sum()) for mm in members], np.int64)
    out = []
    for c in np.argsort(-sums, kind="stable"):
        mm = members[c]
        q = np.zeros(4)
        t = np.zeros(3)
        for k in mm:
            q = q + raw["q"][k]
            t = t + raw["t"][k]
        inv = 1.0 / len(mm)
        q, t = q * inv, t * inv
        nq = math.sqrt(q[0] * q[0] + q[1] * q[1] + q[2] * q[2] + q[3] * q[3])
        if nq > 0:
            q = q / nq
        w, x, y, z = q
        P = np.zeros((4, 4))
        P[0, :3] = 1 - 2 * (y * y + z * z), 2 * (x * y - z * w), 2 * (x * z + y * w)
        P[1, :3] = 2 * (x * y + z * w), 1 - 2 * (x * x + z * z), 2 * (y * z - x * w)
        P[2, :3] = 2 * (x * z - y * w), 2 * (y * z + x * w), 1 - 2 * (x * x + y * y)
        P[:3, 3], P[3, 3] = t, 1.0
        angle, _, _ = update_pose(P[None])
        out.append({"pose": P, "angle": float(angle[0]), "t": t, "q": q, "num_votes": int(min(sums[c], 0xFFFFFFFF)),
                    "leader": leaders[c], "members": mm})
    return out


def match(tr: Trained, scene, relative_scene_sample_step=1.0 / 5.0, relative_scene_distance=0.03, edge=None,
          position_threshold=None, rotation_threshold=None, keep_accumulators=()):
    """match (edge None) / match_S2B as inferred (references from the sampled scene, paired with the sampled edge
    cloud) -> Match; keep_accumulators: reference numbers whose accumulators are returned"""
    margins = Margins()
    sc = sample(scene, np.float32(relative_scene_distance))
    second = sc if edge is None else sample(edge, np.float32(relative_scene_distance))
    step = int(1.0 / relative_scene_sample_step)
    refs = (len(sc) + step - 1) // step
    votes = np.zeros(refs, np.uint32)
    mi = np.zeros(refs, np.uint32)
    ai = np.zeros(refs, np.uint32)
    accs, ties, over, over_refs = {}, 0, {"before_last_row": 0, "last_row": 0}, []
    keep = set(int(r) for r in keep_accumulators)
    for r in range(refs):
        i = r * step
        acc, nb, nl = vote_one(tr, sc[i, :3].astype(np.float64), sc[i, 3:].astype(np.float64), second,
                               i if edge is None else None, margins)
        over["before_last_row"] += nb
        over["last_row"] += nl
        if nb or nl:
            over_refs.append(r)
        flat = int(np.argmax(acc))  # the first maximum in (model point, alpha index) order
        votes[r] = acc.reshape(-1)[flat]
        mi[r], ai[r] = divmod(flat, tr.num_angles)
        ties += int(votes[r] > 0 and np.count_nonzero(acc == votes[r]) > 1)
        if r in keep:
            accs[r] = acc
    P, alpha, angle, t, q = peak_poses(tr, sc[::step][:refs], mi.astype(np.int64), ai, margins)
    raw = {"pose": P.reshape(refs, 16), "alpha": alpha, "angle": angle, "t": t, "q": q, "model_index": mi,
           "num_votes": votes, "alpha_index": ai, "reference_index": np.arange(refs, dtype=np.uint32)}
    pos = tr.position_threshold if position_threshold is None else position_threshold
    rot = tr.rotation_threshold if rotation_threshold is None else rotation_threshold
    clusters = cluster_poses(raw, pos, rot, margins)
    return Match(sc, second, step, raw, clusters, accs, margins, over, over_refs, ties)


# ---- clouds ------------------------------------------------------------------------------------------------------------
def rigid(axis, angle, t):
    axis = np.asarray(axis, np.float64) / np.linalg.norm(axis)
    K = np.array([[0, -axis[2], axis[1]], [axis[2], 0, -axis[0]], [-axis[1], axis[0], 0]])
    T = np.eye(4)
    T[:3, :3] = np.eye(3) + np.sin(angle) * K + (1 - np.cos(angle)) * K @ K
    T[:3, 3] = t
    return T


def moved(cloud, G):
    return np.concatenate([cloud[:, :3] @ G[:3, :3].T + G[:3, 3], cloud[:, 3:6] @ G[:3, :3].T], axis=1)


def bottle_scene(bottle_5mm, n_clutter=600, seed=7):
    """the bottle under a known rigid motion inside normal-distributed clutter, and a curvature-edge-like subset of the
    instance (the points where the profile bends most: the shoulder and the rims) -> (model, scene, edge, G)"""
    G = rigid((0.3, 1.0, 0.2), 0.7, (0.1, -0.05, 0.3))
    rng = np.random.default_rng(seed)
    inst = moved(bottle_5mm, G)
    centre = inst[:, :3].mean(0)
    clutter = np.concatenate([centre + rng.normal(scale=0.15, size=(n_clutter, 3)), rng.normal(size=(n_clutter, 3))], axis=1)
    clutter[:, 3:] /= np.linalg.norm(clutter[:, 3:], axis=1, keepdims=True)
    scene = np.concatenate([inst, clutter]).astype(np.float32)
    z = bottle_5mm[:, :3] @ np.linalg.eigh(np.cov(bottle_5mm[:, :3].T))[1][:, -1]
    q = np.quantile(z, [0.03, 0.62, 0.72, 0.97])
    edge = inst[(z < q[0]) | ((z > q[1]) & (z < q[2])) | (z > q[3])].astype(np.float32)
    return bottle_5mm, scene, edge, G


LATTICE_STEP = 1.0 / 8.5  # ns = 8 cells per axis over the lattice clouds' box [0, 4]^3
_AXES = np.eye(3, dtype=np.float32)


def lattice_overflow(seed=7, zero_normal=False):
    """a cloud with one point per sampling cell (cells of 0.5 over the box [0, 4]^3, pinned by points at both corners)
    and normals along +x, +y or +z, holding pairs (A, A - e_y) whose normals are +x: for them alpha_m = float(pi) =
    pi + 8.7e-8.  The scene is the model turned a quarter about the box's x axis, plus one pair (B, B - e_y + 2^-26 e_z)
    with +x normals in two cells the turn leaves empty: its alpha_s is -pi + 1.5e-8 and its key that of the (A, A - e_y)
    pairs, so their votes get alpha index numAngles, which lands in bin 0 of the next model point's row, or is dropped
    on the last row (the corner (4, 4, 4) is the last sampled point and has such a partner).  zero_normal: one cell
    instead holds two points with opposite normals, whose average normal is 0.  -> (model, scene)"""
    rng = np.random.default_rng(seed)
    taken = np.zeros((8, 8, 8), bool)
    pts, nrm = [], []

    def put(cell, p, n):
        assert not taken[cell], cell
        taken[cell] = True
        pts.append(np.asarray(p, np.float32))
        nrm.append(np.asarray(n, np.float32))

    taken[0, 0, 0] = True  # the corner (0, 0, 0) owns cell 0
    taken[4, 0, 2] = taken[4, 0, 4] = True  # turned, these are the cells (4, 5, 0), (4, 3, 0) of the scene's pair
    for (i, j, k), (u, v, w) in (((2, 5, 0), (0.3, 0.4, 0.2)), ((5, 7, 0), (0.35, 0.15, 0.2)), ((6, 4, 0), (0.1, 0.3, 0.2))):
        a = np.array([0.5 * i + u, 0.5 * j + v, w], np.float32)  # A - e_y is two cells lower in y
        put((i, j, k), a, _AXES[0])
        put((i, j - 2, k), a - np.float32([0, 1, 0]), _AXES[0])
    if zero_normal:
        base = np.float32([1.5, 1.5, 1.5])
        taken[3, 3, 3] = True
        pts += [base + np.float32([0.13, 0.27, 0.31]), base + np.float32([0.36, 0.21, 0.07])]
        nrm += [_AXES[2], -_AXES[2]]
    for cell in zip(*np.nonzero(~taken)):
        if rng.random() < 0.35:
            put(cell, (np.asarray(cell) + rng.uniform(0.15, 0.85, 3)) * 0.5, _AXES[rng.integers(3)])
    pts += [np.float32([0, 0, 0]), np.float32([4, 4, 4]), np.float32([4, 3, 4])]  # (4, 3, 4): cell (8, 6, 8)
    nrm += [_AXES[rng.integers(3)], _AXES[0], _AXES[0]]
    model = np.concatenate([np.stack(pts), np.stack(nrm)], axis=1).astype(np.float32)
    turn = np.array([[1, 0, 0, 0], [0, 0, -1, 4], [0, 1, 0, 0], [0, 0, 0, 1]], np.float64)  # (x, y, z) -> (x, 4 - z, y)
    b = np.float32([2.3, 2.9, 0.2])
    b2 = b - np.float32([0, 1, 0]) + np.float32([0, 0, 2.0 ** -26])
    assert (b2.astype(np.float64) - b.astype(np.float64) == [0, -1, 2.0 ** -26]).all()
    pair = np.array([np.r_[b, _AXES[0]], np.r_[b2, _AXES[0]]], np.float32)
    scene = np.concatenate([moved(model, turn), pair]).astype(np.float32)
    return model, scene


def symmetric_tie(seed=5):
    """a cloud invariant under quarter turns about the x axis ((x, y, z) -> (x, -z, y) is exact in float), every normal
    +x, and a generic rigid motion of it as the scene: symmetric pairs share keys, so peaks tie -> (model, scene)"""
    rng = np.random.default_rng(seed)
    base = np.stack([rng.uniform(-0.1, 0.1, 40), rng.uniform(0.01, 0.1, 40), rng.uniform(0.01, 0.1, 40)], axis=1).astype(np.float32)
    quarter = [base]
    for _ in range(3):
        b = quarter[-1]
        quarter.append(np.stack([b[:, 0], -b[:, 2], b[:, 1]], axis=1))
    xyz = np.concatenate(quarter)
    model = np.concatenate([xyz, np.tile(_AXES[0], (len(xyz), 1))], axis=1).astype(np.float32)
    scene = moved(model, rigid((0.2, -0.5, 1.0), 0.9, (0.05, 0.02, -0.03))).astype(np.float32)
    return model, scene


def over_limit_cloud(n=60000, seed=11):
    """uniform random points and normals in the unit cube: at a relative step of 0.01 they sample to more than
    TABLE_MAX_POINTS points"""
    rng = np.random.default_rng(seed)
    nrm = rng.normal(size=(n, 3))
    nrm /= np.linalg.norm(nrm, axis=1, keepdims=True)
    return np.concatenate([rng.uniform(0, 1, (n, 3)), nrm], axis=1).astype(np.float32)
