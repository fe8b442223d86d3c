"""Own-cell blocks (k2_table.cu own_block_kernel, k3_vote.cu own_step): inside every phase cell the unmerged entries are
stably partitioned by the top OWN_BLOCK_BITS bits of their sub-phase byte, so that a warp step of the scene phase's own
cell whose entries all lie on one side of the scene's own sub-phases votes with one shift.  The partition only makes the
walk faster: the per-step test reads every entry's own byte.  These tests check the layout a build and a load leave, and
the accumulators bit-exact against the oracle on a partitioned table, on the same table left in sorted order, and on a
file whose entries were shuffled inside their cells, with the scene phase placed at block edges and at both ends of its
cell."""
import contextlib
import os

import numpy as np
import pytest

from conftest import ANGLE_STEP, DIST_STEP

pytestmark = pytest.mark.gpu

OWN_BLOCK_BITS = 5  # k2_table.cu
OWN_SUB_MIN = 96    # k3_vote.cu: shorter own cells are compared in full
CELLS = 16
PLANE_Z = np.float32(0.55)  # just below the bottle (z 0.559 ... 0.681)


@contextlib.contextmanager
def sorted_entries():
    """tables built or loaded inside keep each cell's entries in sorted (bin of alpha_m, i, j) order"""
    os.environ["B200PPF_NO_OWN_BLOCKS"] = "1"
    try:
        yield
    finally:
        del os.environ["B200PPF_NO_OWN_BLOCKS"]


class TableFile:
    """the arrays of a saved table: offsets, sub_offsets, entry_w, entry_am, entry_alpha, entry_idx, merged_w, merged cell
    offsets (csrc/capi.cu b200ppf_table_save)"""

    def __init__(self, path):
        self.raw = bytearray(open(path, "rb").read())
        self.hdr = int(np.frombuffer(self.raw[12:16], "<u4")[0])
        n_off, n_sub, n_ent, n_mrg = (int(x) for x in np.frombuffer(self.raw[24:56], "<u8"))
        self.counts = (n_off, n_sub, n_ent, n_ent, n_ent, n_ent, n_mrg, n_sub if n_mrg else 0)
        self.starts = np.cumsum((0,) + self.counts[:-1]) * 4 + self.hdr
        assert self.starts[-1] + 4 * self.counts[-1] == len(self.raw)

    def array(self, k):
        s = int(self.starts[k])
        return np.frombuffer(bytes(self.raw[s:s + 4 * self.counts[k]]), "<u4").copy()

    def put(self, k, a):
        s = int(self.starts[k])
        self.raw[s:s + 4 * self.counts[k]] = np.asarray(a, "<u4").tobytes()

    def write(self, path):
        h = _mix_bytes(0x42323030, self.raw[64:self.hdr])
        for k, cnt in enumerate(self.counts):
            h = _mix_bytes(h, self.raw[int(self.starts[k]):int(self.starts[k]) + 4 * cnt])
        self.raw[56:64] = np.array([h], "<u8").tobytes()
        open(path, "wb").write(bytes(self.raw))


def _mix_bytes(h, data):
    """the table file's 64-bit multiplicative checksum (csrc/capi.cu mix_bytes)"""
    M = (1 << 64) - 1
    data = bytes(data)
    data += b"\0" * (-len(data) % 8)
    for w in np.frombuffer(data, "<u8").tolist():
        h = ((h ^ w) * 0x9E3779B97F4A7C15) & M
        h ^= h >> 29
    return h


def entry_cells(sub):
    return np.repeat(np.arange(len(sub) - 1, dtype=np.int64), np.diff(sub.astype(np.int64)))


def blocks(w, bits=OWN_BLOCK_BITS):
    return (w >> np.uint32(32 - bits)).astype(np.int64)


def stable_blocks_of(tf):
    """the order a stable partition of each cell by block gives to tf's entries"""
    cells = entry_cells(tf.array(1))
    return np.argsort(cells * (1 << OWN_BLOCK_BITS) + blocks(tf.array(2)), kind="stable")


def saved(t, path):
    t.save(str(path))
    return TableFile(str(path))


@pytest.fixture(scope="module")
def tables(ctx, oracle, bottle_5mm, tmp_path_factory):
    """the 2 009-point model's 4 M-entry table (it folds), built with the partition and without it"""
    feats = oracle.ppf_estimation(bottle_5mm)
    hm = oracle.HashMap(ANGLE_STEP, DIST_STEP).set_input_feature_cloud(feats)
    dev_feats = ctx.features_upload(feats)
    t = ctx.table_build(dev_feats, ANGLE_STEP, DIST_STEP)
    with sorted_entries():
        t0 = ctx.table_build(dev_feats, ANGLE_STEP, DIST_STEP)
    assert t.info.n_entries == hm.num_entries >= 1 << 21 and t.info.phase_cells == CELLS
    d = tmp_path_factory.mktemp("own_blocks")
    return t, t0, hm, saved(t, d / "blocks.b200ppf"), saved(t0, d / "sorted.b200ppf"), d


def test_own_blocks_layout(tables):
    """Each cell's blocks are non-decreasing, each block keeps the sorted order, and nothing else moves: the cell bounds,
    the merged words and their bounds are those of the unpartitioned table."""
    _, _, _, tf, tf0, _ = tables
    for k in (0, 1, 6, 7):
        assert np.array_equal(tf.array(k), tf0.array(k)), k
    w0 = tf0.array(2)
    cells = entry_cells(tf.array(1))
    same = cells[1:] == cells[:-1]
    assert np.all(np.diff(blocks(tf.array(2)))[same] >= 0)
    assert np.any(np.diff(blocks(w0))[same] < 0), "the sorted order was already partitioned: the test shows nothing"
    order = stable_blocks_of(tf0)
    for k in (2, 3, 4, 5):
        assert np.array_equal(tf.array(k), tf0.array(k)[order]), k
    # the hard-coded block width is the one the library uses: finer blocks are not ordered any more
    assert np.any(np.diff(blocks(tf.array(2), OWN_BLOCK_BITS + 1))[same] < 0)


def test_small_tables_keep_the_sorted_order(ctx, oracle_bottle, tmp_path):
    """A table too small to fold (the kernel without the one-side test) is left in sorted order, built or loaded."""
    feats, _ = oracle_bottle
    t = ctx.table_build(ctx.features_upload(feats), ANGLE_STEP, DIST_STEP)
    assert t.info.n_entries < 1 << 21 and t.info.phase_cells == CELLS
    with sorted_entries():
        t0 = ctx.table_build(ctx.features_upload(feats), ANGLE_STEP, DIST_STEP)
    tf, tf0 = saved(t, tmp_path / "small.b200ppf"), saved(t0, tmp_path / "small_sorted.b200ppf")
    assert bytes(tf.raw) == bytes(tf0.raw)
    assert bytes(saved(ctx.table_load(str(tmp_path / "small.b200ppf")), tmp_path / "reloaded.b200ppf").raw) == bytes(tf.raw)


def plane_patch(spacing=0.0025, lo=(-0.3, -0.3), hi=(0.2, 0.2)):
    xs = np.arange(lo[0], hi[0], spacing, dtype=np.float64)
    ys = np.arange(lo[1], hi[1], spacing, dtype=np.float64)
    X, Y = np.meshgrid(xs, ys, indexing="ij")
    P = np.zeros((X.size, 6), np.float32)
    P[:, 0], P[:, 1], P[:, 2], P[:, 5] = X.ravel(), Y.ravel(), PLANE_Z, 1.0
    return P


def _rotate_z(P, centre, theta):
    c, s = np.cos(theta), np.sin(theta)
    R = np.array([[c, -s, 0.0], [s, c, 0.0], [0.0, 0.0, 1.0]])
    out = np.empty_like(P)
    out[:, :3] = ((P[:, :3].astype(np.float64) - centre) @ R.T + centre).astype(np.float32)
    out[:, 3:] = (P[:, 3:].astype(np.float64) @ R.T).astype(np.float32)
    return out


def check_acc(ctx, t, hm, n_model, ds, s_r):
    inr, d, a = ctx.vote_debug_pairs(t, ds, s_r)
    acc = ctx.vote_debug_accumulator(t, ds, s_r)
    ref, votes = hm.vote_accumulate_from_pairs(n_model, d[inr > 0], a[inr > 0])
    assert votes == int(acc.sum()), (s_r, votes, int(acc.sum()))
    assert np.array_equal(acc, ref), f"accumulator differs for reference {s_r}"
    return acc


def own_cell_lengths(t, tf, d, a):
    """length of the scene phase's own cell, per in-radius pair and accumulator slice (pairs whose phase sits in a cell)"""
    ti = t.info
    sub = tf.array(1).astype(np.int64)
    lo, size = np.array(ti.lo), np.array(ti.size)
    e = d - lo
    ok = np.all((e >= 0) & (e < size), axis=1)
    key = ((e[:, 3] * size[0] + e[:, 0]) * size[1] + e[:, 1]) * size[2] + e[:, 2]
    u = np.mod(a.astype(np.float64) / float(ANGLE_STEP), 2 * np.pi / float(ANGLE_STEP))
    cell = np.minimum(((u - np.floor(u)) * CELLS).astype(np.int64), CELLS - 1)
    out = []
    for s in range(ti.n_slices):
        c = ((s * ti.key_space + key[ok]) * CELLS + cell[ok])
        out.append(sub[c + 1] - sub[c])
    return np.concatenate(out)


@pytest.fixture(scope="module")
def phase_scene(ctx, bottle_5mm, tables):
    """A plane patch with the bottle on it, plus object points copied around a plane reference point's normal: the pair
    features (so the bucket) stay, the scene phase moves — to block edges inside its cell (the scene's own sub-phases in
    two blocks), just beside them, and to the first and last sub-phase of the cell (sub_lo = 0, sub_hi = 255)."""
    t = tables[0]
    plane = plane_patch()
    n_plane = plane.shape[0]
    s_r = int(np.argmin(np.linalg.norm(plane[:, :2] - np.array([-0.06, -0.05], np.float32), axis=1)))
    centre = plane[s_r, :3].astype(np.float64)
    radius = 0.5 * float(t.info.max_dist)
    dist = np.linalg.norm(bottle_5mm[:, :3] - plane[s_r, :3], axis=1)
    base = bottle_5mm[np.flatnonzero(dist < 0.8 * radius)[::61][:16]]
    assert len(base) >= 8
    probe = np.concatenate([plane, base, _rotate_z(base, centre, 0.01)]).astype(np.float32)
    inr, _, a = ctx.vote_debug_pairs(t, ctx.upload_cloud(probe), s_r)
    a0 = a[n_plane:n_plane + len(base)].astype(np.float64)
    a1 = a[n_plane + len(base):].astype(np.float64)
    assert inr[n_plane:].all()
    sign = np.sign(np.median(a1 - a0))
    step = float(ANGLE_STEP)
    sub_w = 1.0 / (CELLS * 256)  # one sub-phase, in bins
    # positions inside a cell, in sub-phases: every block edge of up to 5 bits, exactly and half a sub-phase to each
    # side, and the first and last sub-phase of the cell
    places = [k * 8 + f for k in range(1, 32) for f in (-0.5, 0.0, 0.5)] + [0.3, 0.6, 255.4, 255.7]
    copies = []
    for i, (b, alpha) in enumerate(zip(base, a0)):
        u = alpha / step
        cell0 = np.floor(u * CELLS) / CELLS
        for p in places[i % 3::3] if len(base) > 3 else places:
            theta = sign * ((cell0 + p * sub_w) * step - alpha)
            copies.append(_rotate_z(b[None], centre, theta))
    scene = np.concatenate([plane, bottle_5mm] + copies).astype(np.float32)
    return scene, s_r, n_plane


def test_own_blocks_accumulators_vs_oracle(ctx, bottle_5mm, tables, phase_scene):
    """Scene phases at block edges and cell ends, dense plane pairs and object pairs: the partitioned table, the same
    table in sorted order (the rule holds in any order) give the oracle's accumulators; both sides of OWN_SUB_MIN occur."""
    t, t0, hm, tf, _, _ = tables
    scene, s_r, n_plane = phase_scene
    ds = ctx.upload_cloud(scene)
    n_model = bottle_5mm.shape[0]
    refs = [s_r, int(np.argmin(np.linalg.norm(scene[:n_plane, :2] - np.array([-0.2, 0.1], np.float32), axis=1))),
            n_plane + 0, n_plane + 1000, n_plane + 2008]
    lengths = []
    for r in refs:
        acc = check_acc(ctx, t, hm, n_model, ds, r)
        assert np.array_equal(check_acc(ctx, t0, hm, n_model, ds, r), acc)
        inr, d, a = ctx.vote_debug_pairs(t, ds, r)
        lengths.append(own_cell_lengths(t, tf, d[inr > 0], a[inr > 0]))
    lengths = np.concatenate(lengths)
    near = lengths[(lengths >= OWN_SUB_MIN - 16) & (lengths < OWN_SUB_MIN + 16)]
    assert np.any(near < OWN_SUB_MIN) and np.any(near >= OWN_SUB_MIN), np.bincount(np.minimum(lengths, 200))
    # the peaks of the partitioned table are those of its accumulators
    hy = ctx.vote(ctx.upload_cloud(bottle_5mm), t, ds, s_r, 1, 2)
    for h in hy:
        acc = ctx.vote_debug_accumulator(t, ds, int(h["scene_index"]))
        flat = int(np.argmax(acc))
        assert h["votes"] == acc.reshape(-1)[flat]


def test_own_blocks_shuffled_file_loads_partitioned(ctx, bottle_5mm, tables, phase_scene):
    """A file whose entries are shuffled inside their cells (any order is a valid table) loads, comes back partitioned —
    stably, so each block keeps the file's order — and votes as the built table does.  A table loaded with the partition
    switched off keeps the file's order and votes the same."""
    t, _, hm, tf, _, d = tables
    rng = np.random.default_rng(7)
    cells = entry_cells(tf.array(1))
    perm = np.lexsort((rng.random(len(cells)), cells))
    shuffled = TableFile(str(d / "blocks.b200ppf"))
    for k in (2, 3, 4, 5):
        shuffled.put(k, tf.array(k)[perm])
    path = str(d / "shuffled.b200ppf")
    shuffled.write(path)
    loaded = ctx.table_load(path)
    tl = saved(loaded, d / "reloaded.b200ppf")
    order = stable_blocks_of(shuffled)
    for k in (2, 3, 4, 5):
        assert np.array_equal(tl.array(k), shuffled.array(k)[order]), k
    assert not np.array_equal(tl.array(5), tf.array(5))
    with sorted_entries():
        as_filed = ctx.table_load(path)
    tf_raw = saved(as_filed, d / "as_filed.b200ppf")
    assert np.array_equal(tf_raw.array(5), shuffled.array(5))
    scene, s_r, _ = phase_scene
    ds = ctx.upload_cloud(scene)
    acc = check_acc(ctx, t, hm, bottle_5mm.shape[0], ds, s_r)
    assert np.array_equal(ctx.vote_debug_accumulator(loaded, ds, s_r), acc)
    assert np.array_equal(ctx.vote_debug_accumulator(as_filed, ds, s_r), acc)
