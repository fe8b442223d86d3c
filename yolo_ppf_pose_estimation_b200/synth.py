"""Seeded synthetic clouds of the shapes BASELINE.json names (SURVEY.md §8d, configs C3-C5).

Host-side workload generators only (numpy); no arithmetic of the PPF path lives here.  The PRNG
is counter-based splitmix64(seed, stream, index), so any language can regenerate the same clouds.

  synth_model(n, seed)  bottle-like closed surface of revolution (z in [0, 0.18] m, r_max 0.05 m,
                        diameter ~0.19 m) with end caps, area-weighted sampling, analytic outward
                        unit normals.
  synth_scene(n, seed)  10 % the model under a ground-truth pose (camera-facing side only), 40 %
                        ground plane, 30 % two walls, 20 % clutter blobs; sigma = 0.5 mm on xyz and
                        2 degrees on normals; normals flipped towards the camera at the origin.
"""
from __future__ import annotations

import numpy as np

_M = np.uint64(0xFFFFFFFFFFFFFFFF)


def splitmix64(x: np.ndarray) -> np.ndarray:
    with np.errstate(over="ignore"):
        x = (x + np.uint64(0x9E3779B97F4A7C15)) & _M
        z = x
        z = ((z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)) & _M
        z = ((z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)) & _M
        return z ^ (z >> np.uint64(31))


def uniform(seed: int, stream: int, n: int) -> np.ndarray:
    """n doubles in [0, 1): splitmix64 of (seed, stream, index)."""
    with np.errstate(over="ignore"):
        base = splitmix64(np.array([seed], np.uint64) * np.uint64(0xD1342543DE82EF95) + np.uint64(stream))
        idx = np.arange(n, dtype=np.uint64)
        bits = splitmix64(base + idx * np.uint64(0x2545F4914F6CDD1D))
    return (bits >> np.uint64(11)).astype(np.float64) * (1.0 / (1 << 53))


def normal(seed: int, stream: int, n: int) -> np.ndarray:
    u1 = np.maximum(uniform(seed, stream, n), 1e-300)
    u2 = uniform(seed, stream + 1, n)
    return np.sqrt(-2.0 * np.log(u1)) * np.cos(2 * np.pi * u2)


# profile of the surface of revolution: (z0, r0) -> (z1, r1) straight segments, bottom to top
_PROFILE = [(0.0, 0.05, 0.11, 0.05), (0.11, 0.05, 0.14, 0.02), (0.14, 0.02, 0.18, 0.02)]


def synth_model(n: int, seed: int = 1, profile: int = 0) -> np.ndarray:
    """(n, 6) float32 [x y z nx ny nz]; profile k scales the shoulder so that a library of models differs."""
    segs = [list(s) for s in _PROFILE]
    if profile:
        segs[1][2] = 0.12 + 0.005 * (profile % 5)   # shoulder height
        segs[2][0] = segs[1][2]
        segs[1][3] = segs[2][1] = segs[2][3] = 0.015 + 0.004 * (profile % 4)  # neck radius
    areas = []
    for z0, r0, z1, r1 in segs:
        slant = np.hypot(z1 - z0, r1 - r0)
        areas.append(np.pi * (r0 + r1) * slant)
    r_bot, r_top = segs[0][1], segs[-1][3]
    areas += [np.pi * r_bot ** 2, np.pi * r_top ** 2]
    cdf = np.cumsum(areas) / np.sum(areas)
    pick = uniform(seed, 0, n)
    u = uniform(seed, 1, n)
    phi = 2 * np.pi * uniform(seed, 2, n)
    part = np.searchsorted(cdf, pick, side="right").clip(0, len(areas) - 1)
    out = np.zeros((n, 6), np.float64)
    for k, (z0, r0, z1, r1) in enumerate(segs):
        m = part == k
        # radius-weighted position along the segment (uniform in area on a cone frustum)
        if abs(r1 - r0) < 1e-12:
            t = u[m]
        else:
            a, b = r0, r1 - r0
            t = (-a + np.sqrt(a * a + u[m] * (2 * a * b + b * b))) / b
        z = z0 + t * (z1 - z0)
        r = r0 + t * (r1 - r0)
        slope = (r1 - r0) / (z1 - z0)
        nn = np.stack([np.cos(phi[m]), np.sin(phi[m]), np.full(m.sum(), -slope)], axis=1)
        nn /= np.linalg.norm(nn, axis=1, keepdims=True)
        out[m, 0], out[m, 1], out[m, 2] = r * np.cos(phi[m]), r * np.sin(phi[m]), z
        out[m, 3:] = nn
    for k, (zc, rc, nz) in enumerate(((0.0, r_bot, -1.0), (segs[-1][2], r_top, 1.0))):
        m = part == len(segs) + k
        r = rc * np.sqrt(u[m])
        out[m, 0], out[m, 1], out[m, 2] = r * np.cos(phi[m]), r * np.sin(phi[m]), zc
        out[m, 5] = nz
    return out.astype(np.float32)


def gt_pose(seed: int = 2) -> np.ndarray:
    """Ground-truth model -> scene pose of synth_scene (4x4 float64)."""
    q = normal(seed, 100, 4)
    q /= np.linalg.norm(q)
    x, y, z, w = q
    R = np.array([[1 - 2 * (y * y + z * z), 2 * (x * y - z * w), 2 * (x * z + y * w)],
                  [2 * (x * y + z * w), 1 - 2 * (x * x + z * z), 2 * (y * z - x * w)],
                  [2 * (x * z - y * w), 2 * (y * z + x * w), 1 - 2 * (x * x + y * y)]])
    T = np.eye(4)
    T[:3, :3] = R
    T[:3, 3] = (0.1, -0.05, 0.9)
    return T


def synth_scene(n: int, seed: int = 2, model_seed: int = 1, model_profile: int = 0,
                model_fraction: float = 0.10) -> np.ndarray:
    """(n, 6) float32 scene containing one instance of synth_model(., model_seed) under gt_pose(seed)."""
    n_model = int(round(model_fraction * n))
    n_ground = int(round(0.40 * n))
    n_wall = int(round(0.30 * n))
    n_clutter = n - n_model - n_ground - n_wall
    parts = []
    # model instance, camera-facing side only
    T = gt_pose(seed)
    cand = synth_model(4 * n_model + 64, model_seed + 7919, model_profile).astype(np.float64)
    p = cand[:, :3] @ T[:3, :3].T + T[:3, 3]
    nn = cand[:, 3:] @ T[:3, :3].T
    facing = np.einsum("ij,ij->i", nn, -p) > 0
    sel = np.flatnonzero(facing)[:n_model]
    if len(sel) < n_model:  # extremely unlikely; pad with back-facing points
        sel = np.concatenate([sel, np.flatnonzero(~facing)[: n_model - len(sel)]])
    parts.append(np.concatenate([p[sel], nn[sel]], axis=1))
    # ground plane y = 0.45 (camera looks along +z, y down), 2 x 2 m
    gx = -1.0 + 2.0 * uniform(seed, 10, n_ground)
    gz = 0.5 + 2.0 * uniform(seed, 11, n_ground)
    g = np.stack([gx, np.full(n_ground, 0.45), gz, np.zeros(n_ground), -np.ones(n_ground), np.zeros(n_ground)], axis=1)
    parts.append(g)
    # two walls: back wall z = 2.5 and side wall x = -1
    nb = n_wall // 2
    bx = -1.0 + 2.0 * uniform(seed, 20, nb)
    by = -0.6 + 1.05 * uniform(seed, 21, nb)
    parts.append(np.stack([bx, by, np.full(nb, 2.5), np.zeros(nb), np.zeros(nb), -np.ones(nb)], axis=1))
    ns = n_wall - nb
    sy = -0.6 + 1.05 * uniform(seed, 22, ns)
    sz = 0.5 + 2.0 * uniform(seed, 23, ns)
    parts.append(np.stack([np.full(ns, -1.0), sy, sz, np.ones(ns), np.zeros(ns), np.zeros(ns)], axis=1))
    # clutter: uniform-in-ball blobs of radius 5 cm, outward normals
    n_blobs = max(1, n_clutter // 400)
    cx = -0.9 + 1.8 * uniform(seed, 30, n_blobs)
    cy = -0.5 + 0.9 * uniform(seed, 31, n_blobs)
    cz = 0.6 + 1.8 * uniform(seed, 32, n_blobs)
    which = (uniform(seed, 33, n_clutter) * n_blobs).astype(np.int64).clip(0, n_blobs - 1)
    d = np.stack([normal(seed, 40, n_clutter), normal(seed, 42, n_clutter), normal(seed, 44, n_clutter)], axis=1)
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    rad = 0.05 * np.cbrt(uniform(seed, 34, n_clutter))
    cp = np.stack([cx[which], cy[which], cz[which]], axis=1) + d * rad[:, None]
    parts.append(np.concatenate([cp, d], axis=1))
    s = np.concatenate(parts, axis=0)
    m = s.shape[0]
    # sensor noise: 0.5 mm on xyz, 2 degrees on normals
    s[:, 0] += 0.0005 * normal(seed, 50, m)
    s[:, 1] += 0.0005 * normal(seed, 52, m)
    s[:, 2] += 0.0005 * normal(seed, 54, m)
    sig = np.radians(2.0)
    s[:, 3] += sig * normal(seed, 60, m)
    s[:, 4] += sig * normal(seed, 62, m)
    s[:, 5] += sig * normal(seed, 64, m)
    s[:, 3:] /= np.linalg.norm(s[:, 3:], axis=1, keepdims=True)
    flip = np.einsum("ij,ij->i", s[:, 3:], -s[:, :3]) < 0
    s[flip, 3:] *= -1
    # fixed pseudo-random order so that reference-point shards see the same mix of surfaces
    order = np.argsort(uniform(seed, 70, m), kind="stable")
    return s[order].astype(np.float32)


def library_pose(k: int, seed: int = 3) -> np.ndarray:
    """Ground-truth pose of library model k in synth_library_scene: rotation from the seed, instances on a 4 x 2 grid."""
    T = gt_pose(seed * 1000 + k)
    T[:3, 3] = (-0.6 + 0.4 * (k % 4), -0.25 + 0.35 * (k // 4), 0.9 + 0.1 * (k % 3))
    return T


def synth_library_scene(n: int = 1 << 20, seed: int = 3, n_models: int = 8, model_points: int = 2000) -> np.ndarray:
    """(n, 6) float32 scene of BASELINE config 4: n = 1024 x 1024 points (the Azure Kinect WFOV-unbinned depth
    size, include/StaticImageProperties.h:65-66 of the reference) holding one camera-facing instance of each of
    the n_models library models synth_model(model_points, 10 + k, profile k) under library_pose(k) — 1.5 % of
    the points each — plus the ground plane, walls and clutter of synth_scene, with the same sensor noise."""
    per_model = int(round(0.015 * n))
    rest = synth_scene(n - n_models * per_model, seed, model_fraction=0.0).astype(np.float64)
    parts = [rest]
    for k in range(n_models):
        T = library_pose(k, seed)
        cand = synth_model(4 * per_model + 64, 10 + k + 7919, k).astype(np.float64)
        p = cand[:, :3] @ T[:3, :3].T + T[:3, 3]
        nn = cand[:, 3:] @ T[:3, :3].T
        sel = np.flatnonzero(np.einsum("ij,ij->i", nn, -p) > 0)[:per_model]
        inst = np.concatenate([p[sel], nn[sel]], axis=1)
        m = inst.shape[0]
        for c in range(3):
            inst[:, c] += 0.0005 * normal(seed, 200 + 10 * k + c, m)
        parts.append(inst)
    s = np.concatenate(parts, axis=0)
    s = s[: n] if s.shape[0] >= n else np.concatenate([s, rest[: n - s.shape[0]]], axis=0)
    order = np.argsort(uniform(seed, 71, s.shape[0]), kind="stable")
    return s[order].astype(np.float32)


DEPTH_SHAPE = (1024, 1024)
DEPTH_K = (400.0, 400.0, 511.5, 511.5)  # fx, fy, ppx, ppy: the 8 library instances all in view
DEPTH_OCCLUDED = (2, 6)  # the library instances a sphere stands in front of: poses whose decoys the unhidden half still tells apart


def _sphere_depth(depth, label, lab, centre, radius, K):
    """render one sphere into depth (z of the nearer intersection per ray; pixel (u, v) looks along ((u - ppx) / fx,
    (v - ppy) / fy, 1)), writing lab into label where it is nearest; only the pixels of its projected bounding square"""
    fx, fy, ppx, ppy = K
    rows, cols = depth.shape
    c = np.asarray(centre, np.float64)
    if c[2] <= radius:
        return
    reach = radius / (c[2] - radius)
    u0 = int(max(0, np.floor(fx * (c[0] / c[2] - reach) + ppx)))
    u1 = int(min(cols - 1, np.ceil(fx * (c[0] / c[2] + reach) + ppx)))
    v0 = int(max(0, np.floor(fy * (c[1] / c[2] - reach) + ppy)))
    v1 = int(min(rows - 1, np.ceil(fy * (c[1] / c[2] + reach) + ppy)))
    if u0 > u1 or v0 > v1:
        return
    v, u = np.mgrid[v0:v1 + 1, u0:u1 + 1]
    wx, wy = (u - ppx) / fx, (v - ppy) / fy
    a = wx * wx + wy * wy + 1.0
    b = -2.0 * (wx * c[0] + wy * c[1] + c[2])
    cc = c @ c - radius * radius
    disc = b * b - 4 * a * cc
    hit = disc >= 0
    t = np.where(hit, (-b - np.sqrt(np.where(hit, disc, 0))) / (2 * a), np.inf)
    sub, lsub = depth[v0:v1 + 1, u0:u1 + 1], label[v0:v1 + 1, u0:u1 + 1]
    near = hit & (t > 0) & (t < sub)
    sub[near] = t[near]
    lsub[near] = lab


def synth_library_depth(seed: int = 3, n_models: int = 8, dense: int = 300_000, occluded=DEPTH_OCCLUDED):
    """A deterministic depth frame of the library scene: DEPTH_SHAPE float32 metres under DEPTH_K, holding the ground plane
    and walls of synth_scene (intersected per ray), its clutter spheres (radius 5 cm) except those whose image disc meets an
    instance's box, the n_models library instances under library_pose(k) (a dense synth_model(dense, 10 + k + 7919, k)
    splatted one point per pixel, nearest wins) and, in front of each instance of `occluded`, a sphere covering 30-60 % of
    that instance's visible pixels on the side of its base.  0.5 mm of sensor noise on every measured depth; rays that meet nothing read 0.
    -> dict(depth, K (4,), occluded_share (n_models,), occluders [(k, centre, radius)])"""
    rows, cols = DEPTH_SHAPE
    fx, fy, ppx, ppy = DEPTH_K
    v, u = np.mgrid[0:rows, 0:cols]
    wx, wy = (u - ppx) / fx, (v - ppy) / fy
    depth = np.full(DEPTH_SHAPE, np.inf)
    label = np.full(DEPTH_SHAPE, -1, np.int64)  # -1 background, k instance k, n_models + j occluder j
    with np.errstate(divide="ignore", invalid="ignore"):
        t = 0.45 / wy  # ground y = 0.45, x in [-1, 1], z in [0.5, 2.5]
        ok = (wy > 0) & (np.abs(t * wx) <= 1.0) & (t >= 0.5) & (t <= 2.5)
        depth[ok] = np.minimum(depth[ok], t[ok])
        t = np.full(DEPTH_SHAPE, 2.5)  # back wall z = 2.5, x in [-1, 1], y in [-0.6, 0.45]
        ok = (np.abs(t * wx) <= 1.0) & (t * wy >= -0.6) & (t * wy <= 0.45)
        depth[ok] = np.minimum(depth[ok], t[ok])
        t = -1.0 / wx  # side wall x = -1, y in [-0.6, 0.45], z in [0.5, 2.5]
        ok = (wx < 0) & (t * wy >= -0.6) & (t * wy <= 0.45) & (t >= 0.5) & (t <= 2.5)
        depth[ok] = np.minimum(depth[ok], t[ok])
    # the instances, one dense splat each, and their image boxes
    boxes = []
    for k in range(n_models):
        T = library_pose(k, seed)
        m = synth_model(dense, 10 + k + 7919, k).astype(np.float64)
        p = m[:, :3] @ T[:3, :3].T + T[:3, 3]
        pu = np.floor(fx * p[:, 0] / p[:, 2] + ppx + 0.5).astype(np.int64)
        pv = np.floor(fy * p[:, 1] / p[:, 2] + ppy + 0.5).astype(np.int64)
        inside = (pu >= 0) & (pu < cols) & (pv >= 0) & (pv < rows)
        pu, pv, pz = pu[inside], pv[inside], p[inside, 2]
        boxes.append((pu.min(), pu.max(), pv.min(), pv.max()))
        flat = depth.ravel()
        lab = label.ravel()
        before = flat.copy()
        np.minimum.at(flat, pv * cols + pu, pz)
        lab[flat < before] = k
    # the clutter spheres of synth_scene (synth_library_scene's share of the points), away from the instances
    n_rest = (1 << 20) - n_models * int(round(0.015 * (1 << 20)))
    n_clutter = n_rest - int(round(0.40 * n_rest)) - int(round(0.30 * n_rest))
    n_blobs = max(1, n_clutter // 400)
    cs = np.stack([-0.9 + 1.8 * uniform(seed, 30, n_blobs), -0.5 + 0.9 * uniform(seed, 31, n_blobs),
                   0.6 + 1.8 * uniform(seed, 32, n_blobs)], 1)
    for c in cs:
        reach = 0.05 / (c[2] - 0.05)
        cu0, cu1 = fx * (c[0] / c[2] - reach) + ppx, fx * (c[0] / c[2] + reach) + ppx
        cv0, cv1 = fy * (c[1] / c[2] - reach) + ppy, fy * (c[1] / c[2] + reach) + ppy
        if any(cu1 >= b[0] - 2 and cu0 <= b[1] + 2 and cv1 >= b[2] - 2 and cv0 <= b[3] + 2 for b in boxes):
            continue
        _sphere_depth(depth, label, -1, c, 0.05, DEPTH_K)
    # the occluders: a sphere 25 cm in front of the instance, moved from its centre toward its base until it hides at most
    # half of it; the shoulder and neck, which tell a pose from its shifted and upside-down twins, stay in view
    share = np.zeros(n_models)
    occluders = []
    for j, k in enumerate(occluded):
        mine = label == k
        vv, uu = np.nonzero(mine)
        zc = float(np.median(depth[mine]))
        ray = np.array([(uu.mean() - ppx) / fx, (vv.mean() - ppy) / fy, 1.0])
        zo, radius = zc - 0.25, 0.05
        base = library_pose(k, seed)[:3, 3]  # the model's origin: the centre of its base
        toward = base / base[2] - ray
        toward = np.array([toward[0], toward[1], 0.0]) / np.hypot(toward[0], toward[1])
        for shift in np.arange(0.0, 0.2, 0.004):
            centre = ray * zo + shift * toward
            d2, l2 = depth.copy(), label.copy()
            _sphere_depth(d2, l2, n_models + j, centre, radius, DEPTH_K)
            s = float(((l2 == n_models + j) & mine).sum()) / mine.sum()
            if s <= 0.5:
                break
        assert 0.3 <= s <= 0.6, (k, s)
        depth, label = d2, l2
        share[k] = s
        occluders.append((k, centre, radius))
    measured = np.isfinite(depth)
    noisy = depth + 0.0005 * normal(seed, 300, rows * cols).reshape(DEPTH_SHAPE)
    out = np.where(measured, noisy, 0.0).astype(np.float32)
    return dict(depth=out, K=np.array(DEPTH_K, np.float64), occluded_share=share, occluders=occluders)
