"""GPU parity tests: every stage of the CUDA path, through the C ABI, against the CPU oracle.

Fixtures are the reference's own data frozen under tests/golden (tools/make_fixtures.py); nothing
here reads /root/reference.  Rules and tolerances: tests/parity.py.
"""
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ANGLE_STEP, DIST_STEP, ROOT
import parity

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def dev_bottle(ctx, bottle):
    return ctx.upload_cloud(bottle)


@pytest.fixture(scope="module")
def dev_crop(ctx, scene_crop):
    return ctx.upload_cloud(scene_crop)


@pytest.fixture(scope="module")
def table_from_oracle_features(ctx, oracle_bottle):
    """PPFHashMapSearch::setInputFeatureCloud on the oracle's own signatures: identical floats in."""
    feats, _ = oracle_bottle
    return ctx.table_build(ctx.features_upload(feats), ANGLE_STEP, DIST_STEP)


@pytest.fixture(scope="module")
def table_fused(ctx, dev_bottle):
    return ctx.table_build_from_cloud(dev_bottle, ANGLE_STEP, DIST_STEP)


# ---- K1 ------------------------------------------------------------------------------------------

def test_k1_features_vs_oracle(ctx, bottle, dev_bottle, oracle_bottle):
    feats, _ = oracle_bottle
    F = ctx.features_compute(dev_bottle)
    assert F.count == bottle.shape[0] ** 2
    rep = parity.compare_features(bottle, F.download(), feats, ANGLE_STEP, DIST_STEP)
    print("K1 parity:", rep)
    assert rep["swap_ambiguous"] < 50 and rep["key_flips"] < 200


@pytest.mark.parametrize("mode", [1, 2])
def test_k1_drost_modes(bottle, oracle, mode):
    from yolo_ppf_pose_estimation_b200 import capi
    c = capi.Context(0, feature_mode=mode)
    sub = bottle[::4]
    F = c.features_compute(c.upload_cloud(sub)).download()
    ref = oracle.ppf_estimation(sub, mode=mode)
    assert np.array_equal(np.isnan(F[:, 0]), np.isnan(ref[:, 0]))
    v = ~np.isnan(ref[:, 0])
    assert np.array_equal(F[v, 3], ref[v, 3])
    assert np.abs(F[v, :3].astype(np.float64) - ref[v, :3]).max() < 4e-6
    vi = np.flatnonzero(v)
    atol = parity.alpha_tolerance(sub, vi // len(sub), vi % len(sub))
    assert (parity.circ_diff(F[v, 4], ref[v, 4]) <= atol).all()


def test_k1_partial_download_and_bounds(ctx, dev_bottle):
    F = ctx.features_compute(dev_bottle)
    n = dev_bottle.size
    row7 = F.download(7 * n, n)
    assert np.isnan(row7[7]).all() and not np.isnan(row7[8]).any()
    from yolo_ppf_pose_estimation_b200.capi import B200PPFError
    with pytest.raises(B200PPFError):
        F.download(n * n - 1, 2)


# ---- K2 ------------------------------------------------------------------------------------------

def test_k2_buckets_bit_exact(oracle_bottle, table_from_oracle_features):
    """Same signatures in -> identical keys, bucket contents in canonical (i, j) order, alpha_m, diameter."""
    feats, hm = oracle_bottle
    t = table_from_oracle_features
    ti = t.info
    assert ti.n_entries == hm.num_entries == 294306
    assert ti.n_keys == hm.num_keys == 10448
    assert np.float32(ti.max_dist) == np.float32(hm.model_diameter)
    assert ti.n_alpha == 30 and ti.nalpha_rule == 0 and ti.n_slices == 1   # ceil(2*pi / float(12 deg)): the default column rule
    buckets = parity.table_buckets(t)
    keys, lengths = hm.dump_keys()
    assert len(buckets) == len(keys)
    n = ti.n_model
    for key, length in zip(keys, lengths):
        bi, bj, ba = buckets[tuple(int(x) for x in key)]
        ref = hm.query_key(key)
        assert length == len(bi)
        assert np.array_equal(bi, ref[:, 0].astype(np.uint32)) and np.array_equal(bj, ref[:, 1].astype(np.uint32))
        assert np.array_equal(ba.view(np.uint32), feats[bi.astype(np.int64) * n + bj, 4].view(np.uint32))


def test_k2_nearest_neighbor_search(oracle_bottle, table_from_oracle_features):
    feats, hm = oracle_bottle
    rng = np.random.default_rng(3)
    valid = np.flatnonzero(~np.isnan(feats[:, 0]))
    for p in rng.choice(valid, 20, replace=False):
        f = feats[p]
        got = table_from_oracle_features.query(*[float(x) for x in f[:4]])
        want = hm.query(*[float(x) for x in f[:4]])
        assert np.array_equal(got, want)
    # a feature no model pair has -> empty
    assert len(table_from_oracle_features.query(0.0, 0.0, 0.0, 10.0)) == 0
    assert len(table_from_oracle_features.query(float("nan"), 0.0, 0.0, 0.1)) == 0


def test_k2_alpha_m_matrix(oracle_bottle, table_from_oracle_features):
    feats, _ = oracle_bottle
    n = table_from_oracle_features.info.n_model
    A = table_from_oracle_features.alpha_m()
    ref = feats[:, 4].reshape(n, n)
    assert np.array_equal(np.isnan(A), np.isnan(ref))
    assert np.array_equal(A[~np.isnan(ref)].view(np.uint32), ref[~np.isnan(ref)].view(np.uint32))


def test_k2_fused_equals_two_step(ctx, dev_bottle, table_fused):
    """K1+K2 fused build == compute() then setInputFeatureCloud() on the device's own signatures."""
    two = ctx.table_build(ctx.features_compute(dev_bottle), ANGLE_STEP, DIST_STEP)
    a, b = parity.table_buckets(table_fused), parity.table_buckets(two)
    assert a.keys() == b.keys()
    for k in a:
        assert all(np.array_equal(x.view(np.uint32), y.view(np.uint32)) for x, y in zip(a[k], b[k]))
    assert table_fused.info.n_entries == two.info.n_entries
    assert table_fused.info.max_dist == two.info.max_dist


def test_k2_fused_vs_oracle_key_rule(bottle, oracle_bottle, table_fused):
    """Device-computed keys vs oracle keys: flips only within 1e-5 of a bin edge."""
    feats, hm = oracle_bottle
    n = bottle.shape[0]
    off, ei, ej, ea = table_fused.export()
    ti = table_fused.info
    assert ti.n_slices == 1
    lens = np.diff(off.astype(np.int64))
    packed = np.repeat(np.arange(ti.key_space), lens)
    dev_keys = table_fused.unpack_key(packed)
    idx = ei.astype(np.int64) * n + ej
    assert len(np.unique(idx)) == len(idx) == ti.n_entries == hm.num_entries
    ref_keys = parity.quantise(feats[idx, :4], ANGLE_STEP, DIST_STEP)
    flip = dev_keys != ref_keys
    edge = parity.near_edge(feats[idx, :4], ANGLE_STEP, DIST_STEP)
    amb = parity.swap_margin(bottle, ei.astype(np.int64), ej.astype(np.int64)) < parity.EDGE_TOL
    assert not ((flip & ~edge).any(axis=1) & ~amb).any()
    assert flip.any(axis=1).sum() < 200
    assert np.float32(ti.max_dist) == np.float32(hm.model_diameter)


def test_k2_sliced_table_same_buckets(bottle, oracle_bottle):
    """Forcing several accumulator slices must not change bucket contents."""
    code = f"""
import sys, numpy as np
sys.path.insert(0, {ROOT!r}); sys.path.insert(0, {os.path.join(ROOT, 'tests')!r})
from yolo_ppf_pose_estimation_b200 import capi
import parity
from conftest import ANGLE_STEP, DIST_STEP, load_cloud
from oracle import binding as ob
m = load_cloud('bottle_1cm'); s = load_cloud('scene_crop_1cm')
feats = ob.ppf_estimation(m)
c = capi.Context(0)
t = c.table_build(c.features_upload(feats), ANGLE_STEP, DIST_STEP)
assert t.info.n_slices == 4, t.info.n_slices
hm = ob.HashMap(ANGLE_STEP, DIST_STEP).set_input_feature_cloud(feats)
b = parity.table_buckets(t)
keys, lengths = hm.dump_keys()
assert len(b) == len(keys)
for key in keys:
    bi, bj, ba = b[tuple(int(x) for x in key)]
    ref = hm.query_key(key)
    assert np.array_equal(bi, ref[:,0].astype(np.uint32)) and np.array_equal(bj, ref[:,1].astype(np.uint32))
dm, ds = c.upload_cloud(m), c.upload_cloud(s)
for s_r in (0, 401, 933):
    inr, d, a = c.vote_debug_pairs(t, ds, s_r)
    acc = c.vote_debug_accumulator(t, ds, s_r)
    ref, votes = hm.vote_accumulate_from_pairs(m.shape[0], d[inr > 0], a[inr > 0])
    assert np.array_equal(acc, ref), s_r
hy = c.vote(dm, t, ds, 0, 5)
for h in hy[::17]:
    acc = c.vote_debug_accumulator(t, ds, int(h['scene_index']))
    flat = int(np.argmax(acc)); assert h['votes'] == acc.reshape(-1)[flat]
    assert (h['model_index'], h['alpha_bin']) == divmod(flat, acc.shape[1]) or h['votes'] == 0
print('SLICED_OK')
"""
    env = dict(os.environ, B200PPF_SLICE_ROWS="150")
    r = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=600)
    assert "SLICED_OK" in r.stdout, r.stdout + r.stderr


def test_k2_table_save_load(tmp_path, ctx, dev_bottle, dev_crop, table_fused):
    """LoadTrainedDetector path: a saved table reloads to the same buckets and the same votes; corrupt,
    truncated, foreign and mode-mismatched files are refused."""
    from yolo_ppf_pose_estimation_b200 import capi
    path = str(tmp_path / "bottle.b200ppf")
    table_fused.save(path)
    t2 = ctx.table_load(path)
    a, b = table_fused.info, t2.info
    for f, _ in capi.TableInfo._fields_:
        va, vb = getattr(a, f), getattr(b, f)
        assert (list(va) == list(vb)) if hasattr(va, "__len__") else (va == vb), f
    ba, bb = parity.table_buckets(table_fused), parity.table_buckets(t2)
    assert ba.keys() == bb.keys()
    for k in ba:
        assert all(np.array_equal(x.view(np.uint32), y.view(np.uint32)) for x, y in zip(ba[k], bb[k]))
    h1 = ctx.vote(dev_bottle, table_fused, dev_crop, 0, 5)
    h2 = ctx.vote(dev_bottle, t2, dev_crop, 0, 5)
    assert h1.tobytes() == h2.tobytes()
    raw = open(path, "rb").read()
    bad = tmp_path / "bad.b200ppf"
    for blob, msg in ((raw[:len(raw) // 2], "truncated"), (raw + b"x", "trailing"), (b"PLY" + raw[3:], "not a b200ppf"),
                      (raw[:-9] + bytes([raw[-9] ^ 1]) + raw[-8:], "checksum")):
        bad.write_bytes(blob)
        with pytest.raises(capi.B200PPFError) as e:
            ctx.table_load(str(bad))
        assert msg in str(e.value), (msg, str(e.value))
    with pytest.raises(capi.B200PPFError):
        ctx.table_load(str(tmp_path / "missing.b200ppf"))
    cb = capi.Context(0, alpha_mode=capi.ALPHA_MODE_B)
    with pytest.raises(capi.B200PPFError) as e:
        cb.table_load(path)
    assert "mode differs" in str(e.value)


def _mix_bytes(h, data):
    """the table file's 64-bit multiplicative checksum (csrc/capi.cu mix_bytes)"""
    M = (1 << 64) - 1
    data = bytes(data)
    data += b"\0" * (-len(data) % 8)
    for w in np.frombuffer(data, "<u8").tolist():
        h = ((h ^ w) * 0x9E3779B97F4A7C15) & M
        h ^= h >> 29
    return h


def test_k2_table_load_refuses_consistent_looking_but_invalid_files(tmp_path, ctx, dev_bottle):
    """A file whose checksum is RIGHT but whose contents would send the voting kernel out of bounds (rewritten or
    crafted): decreasing offsets, a hot word pointing outside the accumulator slice, a pair index beyond n*n, key
    ranges whose product is not the key space, binning parameters that do not follow from the angle step."""
    import ctypes as C
    from yolo_ppf_pose_estimation_b200 import capi
    small = ctx.upload_cloud(dev_bottle.download()[::6].copy())
    t = ctx.table_build_from_cloud(small, ANGLE_STEP, DIST_STEP)
    path = str(tmp_path / "t.b200ppf")
    t.save(path)
    raw = bytearray(open(path, "rb").read())
    hdr = int(np.frombuffer(raw[12:16], "<u4")[0])
    n_off, n_sub, n_ent, n_mrg = (int(x) for x in np.frombuffer(raw[24:56], "<u8"))
    info_off, info_len = 64, C.sizeof(capi.TableInfo)
    a_off = hdr     # arrays: offsets, sub_offsets, entry_w, entry_am, entry_alpha, entry_idx, merged_w, merged cell offsets
    counts = (n_off, n_sub, n_ent, n_ent, n_ent, n_ent, n_mrg, n_sub if n_mrg else 0)
    starts = np.cumsum((0,) + counts[:-1]) * 4 + a_off
    assert starts[-1] + 4 * counts[-1] == len(raw) and n_mrg and n_mrg < n_ent

    def resign(blob):
        h = _mix_bytes(0x42323030, blob[info_off:hdr])      # info, key and binning parameters
        for k, cnt in enumerate(counts):
            h = _mix_bytes(h, blob[starts[k]:starts[k] + 4 * cnt])
        blob[56:64] = np.array([h], "<u8").tobytes()
        return blob

    good = tmp_path / "good.b200ppf"
    good.write_bytes(resign(bytearray(raw)))
    assert bytes(resign(bytearray(raw))) == bytes(raw)      # the test's checksum is the library's
    ctx.table_load(str(good))

    def word(blob, array, index):
        o = int(starts[array]) + 4 * index
        return o, int(np.frombuffer(blob[o:o + 4], "<u4")[0])

    cases = []
    b = bytearray(raw)                                     # offsets decrease in the middle
    o, v = word(b, 0, n_off // 2)
    b[o:o + 4] = np.array([v + 7], "<u4").tobytes()
    cases.append(("offsets", b))
    b = bytearray(raw)                                     # a hot word far outside the accumulator slice
    o, v = word(b, 2, n_ent // 3)
    b[o:o + 4] = np.array([(v & 0xFF000000) | 0x00FFFFF0], "<u4").tobytes()
    cases.append(("hot word", b))
    b = bytearray(raw)                                     # a merged vote word far outside the accumulator slice
    o, v = word(b, 6, n_mrg // 2)
    b[o:o + 4] = np.array([(v & 0xFF000000) | 0x00FFFFF0], "<u4").tobytes()
    cases.append(("merged vote word", b))
    b = bytearray(raw)                                     # a merged count that no longer matches the cell's entries
    o, v = word(b, 6, n_mrg // 3)
    b[o:o + 4] = np.array([v + (1 << 24)], "<u4").tobytes()
    cases.append(("merged vote counts", b))
    b = bytearray(raw)                                     # pair index beyond n*n
    o, v = word(b, 5, 5)
    b[o:o + 4] = np.array([0x7FFFFFFF], "<u4").tobytes()
    cases.append(("pair index", b))
    b = bytearray(raw)                                     # key ranges: size[0] + 1 (both copies), key_space unchanged
    ti = capi.TableInfo.from_buffer_copy(bytes(raw[info_off:info_off + info_len]))
    ti.size[0] += 1
    b[info_off:info_off + info_len] = bytes(ti)
    kp_size0 = info_off + info_len + 8 + 16                # KeyParams: two float steps, lo[4], size[4], ...
    assert np.frombuffer(b[kp_size0:kp_size0 + 4], "<i4")[0] == ti.size[0] - 1
    b[kp_size0:kp_size0 + 4] = np.array([ti.size[0]], "<i4").tobytes()
    cases.append(("key space", b))
    b = bytearray(raw)                                     # binning: another fixed-point multiplier
    o = info_off + info_len + 4 * 15 + 4 * 10              # KeyParams is 15 words; fix_mul is word 10 of BinParams
    fix_mul = int(np.frombuffer(bytes(raw[o:o + 4]), "<u4")[0])
    T = 2 * np.pi / float(ANGLE_STEP)
    assert any(fix_mul == int(np.rint(T * 2 ** sh)) for sh in range(20, 31)), "header layout changed: update this test"
    b[o:o + 4] = np.array([fix_mul ^ 0x3039], "<u4").tobytes()
    cases.append(("binning parameters", b))
    for what, blob in cases:
        bad = tmp_path / "bad.b200ppf"
        bad.write_bytes(resign(blob))
        with pytest.raises(capi.B200PPFError) as e:
            ctx.table_load(str(bad))
        assert "invalid table" in str(e.value) and what in str(e.value), (what, str(e.value))


@pytest.mark.parametrize("rule", [0, 1, 2])
def test_k3_alpha_column_rules(bottle, scene_crop, oracle, oracle_bottle, rule):
    """The three rules for the accumulator's alpha columns (include/b200ppf.h B200PPF_NALPHA_*): ceil = 30 columns for
    PCL's 12 degrees (default), floor + drop and floor + clamp = 29.  Accumulators bit-exact against the oracle under the
    same rule, hypotheses equal to the oracle's on the same accumulators, the rule survives save / load."""
    from yolo_ppf_pose_estimation_b200 import capi
    feats, _ = oracle_bottle
    hm = oracle.HashMap(ANGLE_STEP, DIST_STEP, nalpha_rule=rule).set_input_feature_cloud(feats)
    c = capi.Context(0, nalpha_rule=rule)
    t = c.table_build(c.features_upload(feats), ANGLE_STEP, DIST_STEP)
    assert t.info.n_alpha == (30 if rule == 0 else 29) == oracle.num_alpha_bins(ANGLE_STEP, rule) and t.info.nalpha_rule == rule
    dm, ds = c.upload_cloud(bottle), c.upload_cloud(scene_crop)
    cast = {}
    for s_r in REFS:
        inr, d, a = c.vote_debug_pairs(t, ds, s_r)
        acc = c.vote_debug_accumulator(t, ds, s_r)
        ref, votes = hm.vote_accumulate_from_pairs(bottle.shape[0], d[inr > 0], a[inr > 0])
        assert acc.shape == ref.shape and np.array_equal(acc, ref), (rule, s_r)
        assert int(acc.sum()) == votes if rule != 1 else int(acc.sum()) < votes    # dropped votes are cast but not stored
        assert c.vote_stats()["votes"] == votes
    hy = c.vote(dm, t, ds, 0, 5)
    for h in hy[::9]:
        acc = c.vote_debug_accumulator(t, ds, int(h["scene_index"]))
        flat = int(np.argmax(acc))
        assert h["votes"] == acc.reshape(-1)[flat]
        if h["votes"]:
            assert (int(h["model_index"]), int(h["alpha_bin"])) == divmod(flat, acc.shape[1])
    import tempfile
    with tempfile.TemporaryDirectory() as d_:
        path = os.path.join(d_, "t.b200ppf")
        t.save(path)
        t2 = capi.Context(0).table_load(path)          # the rule travels with the file, whatever the loading context's is
        assert t2.info.nalpha_rule == rule and t2.info.n_alpha == t.info.n_alpha


# ---- K3 ------------------------------------------------------------------------------------------

REFS = (0, 5, 250, 600, 933)


def test_k3_scene_pairs_vs_oracle(ctx, scene_crop, dev_crop, oracle_bottle, table_from_oracle_features):
    _, hm = oracle_bottle
    radius = np.float32(hm.model_diameter) * np.float32(0.5)
    for s_r in REFS:
        inr, d, a = ctx.vote_debug_pairs(table_from_oracle_features, dev_crop, s_r)
        rin, rd, ra = hm.scene_pairs(scene_crop, s_r)
        dist = np.linalg.norm(scene_crop[:, :3].astype(np.float64) - scene_crop[s_r, :3], axis=1)
        radius_edge = np.abs(dist - float(radius)) < parity.EDGE_TOL
        assert np.array_equal(inr[~radius_edge], rin[~radius_edge])
        both = (inr > 0) & (rin > 0)
        idx_both = np.flatnonzero(both)
        atol = parity.alpha_tolerance(scene_crop, np.full(len(idx_both), s_r), idx_both)
        assert (parity.circ_diff(a[both], ra[both]) <= atol).all()
        flip = (d[both] != rd[both])
        if flip.any():
            # recompute the oracle's float features for the flipped pairs and apply the edge rule
            idx = np.flatnonzero(both)[flip.any(axis=1)]
            for s in idx:
                ok, f = oracle_pair(scene_crop, s_r, s)
                amb = parity.swap_margin(scene_crop, np.array([s_r]), np.array([s]))[0] < parity.EDGE_TOL
                edge = parity.near_edge(f, ANGLE_STEP, DIST_STEP)
                assert amb or not ((d[s] != rd[s]) & ~edge).any(), (s_r, s, f, d[s], rd[s])
        assert flip.any(axis=1).mean() < 0.02


def oracle_pair(cloud, a, b):
    from oracle import binding as ob
    return ob.pair_feature(cloud[a, :3], cloud[a, 3:], cloud[b, :3], cloud[b, 3:])


def test_k3_accumulator_bit_exact(ctx, bottle, dev_crop, oracle_bottle, table_from_oracle_features):
    """Index half of the voting loop: with the device's own per-pair (key, alpha_s) the oracle's
    bucket walk + alpha binning must reproduce the device accumulator exactly."""
    _, hm = oracle_bottle
    for s_r in REFS:
        inr, d, a = ctx.vote_debug_pairs(table_from_oracle_features, dev_crop, s_r)
        acc = ctx.vote_debug_accumulator(table_from_oracle_features, dev_crop, s_r)
        ref, votes = hm.vote_accumulate_from_pairs(bottle.shape[0], d[inr > 0], a[inr > 0])
        assert votes == int(acc.sum())
        assert np.array_equal(acc, ref), f"accumulator differs for reference {s_r}"


def test_k3_accumulator_vs_oracle_floats(ctx, bottle, scene_crop, dev_crop, oracle_bottle, table_from_oracle_features):
    """Whole loop vs the oracle (its own floats): counts may differ only through edge pairs."""
    _, hm = oracle_bottle
    for s_r in REFS:
        acc = ctx.vote_debug_accumulator(table_from_oracle_features, dev_crop, s_r).astype(np.int64)
        ref, votes = hm.vote_accumulate(bottle.shape[0], scene_crop, s_r)
        l1 = np.abs(acc - ref.astype(np.int64)).sum()
        assert l1 <= 0.01 * max(votes, 1) + 8, (s_r, l1, votes)


def test_k3_hypotheses(ctx, bottle, scene_crop, dev_bottle, dev_crop, oracle, oracle_bottle, table_from_oracle_features):
    _, hm = oracle_bottle
    hy = ctx.vote(dev_bottle, table_from_oracle_features, dev_crop, 0, 5)
    ref, stats = hm.vote(bottle, scene_crop, 0, 5, n_threads=oracle.max_threads())
    assert len(hy) == len(ref) == (scene_crop.shape[0] + 4) // 5
    assert np.array_equal(hy["scene_index"], ref["scene_index"])
    st = ctx.vote_stats()
    # candidates met in the 27-cell neighbourhoods: at least the in-radius ones, far fewer than brute force
    assert st["pairs_in_radius"] <= st["pairs_examined"] < len(hy) * (scene_crop.shape[0] - 1)
    assert abs(st["pairs_in_radius"] - stats["pairs_in_radius"]) <= 0.001 * stats["pairs_in_radius"] + 2
    assert abs(st["votes"] - stats["votes"]) <= 0.002 * stats["votes"]
    same_peak = (hy["model_index"] == ref["model_index"]) & (hy["alpha_bin"] == ref["alpha_bin"])
    assert same_peak.mean() > 0.9, same_peak.mean()
    dv = np.abs(hy["votes"].astype(np.int64) - ref["votes"].astype(np.int64))
    assert (dv <= 0.05 * ref["votes"] + 3).all()
    assert (hy["votes"][same_peak] == ref["votes"][same_peak]).mean() > 0.8
    # same peak -> same pose up to libm ulps
    dp = np.abs(hy["pose"][same_peak] - ref["pose"][same_peak]).max()
    assert dp < 2e-5, dp
    # the peak is the first maximum of the device's own accumulator (PCL tie-break)
    for h in hy[::23]:
        acc = ctx.vote_debug_accumulator(table_from_oracle_features, dev_crop, int(h["scene_index"]))
        flat = int(np.argmax(acc))
        assert h["votes"] == acc.reshape(-1)[flat]
        if h["votes"]:
            assert (int(h["model_index"]), int(h["alpha_bin"])) == divmod(flat, acc.shape[1])
        # and its pose is the oracle's pose for that peak
        P = oracle.peak_pose(bottle, int(h["model_index"]), int(h["alpha_bin"]), scene_crop, int(h["scene_index"]),
                             ANGLE_STEP)
        assert np.abs(P.reshape(-1) - h["pose"]).max() < 2e-5


def test_k3_sharding_invariance(ctx, dev_bottle, dev_crop, table_fused):
    """Reference points are independent: any split of the index set gives the same records."""
    full = ctx.vote(dev_bottle, table_fused, dev_crop, 0, 1)
    n = len(full)
    parts = []
    for g in range(4):
        lo, hi = g * n // 4, (g + 1) * n // 4
        parts.append(ctx.vote(dev_bottle, table_fused, dev_crop, lo, 1, hi - lo))
    cat = np.concatenate(parts)
    assert cat.tobytes() == full.tobytes()
    strided = ctx.vote(dev_bottle, table_fused, dev_crop, 3, 7)
    assert strided.tobytes() == full[3::7].tobytes()


def test_k3_large_model_two_slices(ctx, oracle, bottle_5mm, scene_crop, dev_crop):
    """2 009-point bottle: two accumulator slices of ~1 000 rows, the 1024-thread launch shape, long
    buckets (the constant-shift ranges dominate).  Accumulators bit-exact, peaks first-maximum."""
    feats = oracle.ppf_estimation(bottle_5mm)
    hm = oracle.HashMap(ANGLE_STEP, DIST_STEP).set_input_feature_cloud(feats)
    t = ctx.table_build(ctx.features_upload(feats), ANGLE_STEP, DIST_STEP)
    assert t.info.n_slices == 2 and t.info.phase_cells == 16 and t.info.n_entries == hm.num_entries
    for s_r in (0, 433, 933):
        inr, d, a = ctx.vote_debug_pairs(t, dev_crop, s_r)
        acc = ctx.vote_debug_accumulator(t, dev_crop, s_r)
        ref, votes = hm.vote_accumulate_from_pairs(bottle_5mm.shape[0], d[inr > 0], a[inr > 0])
        assert votes == int(acc.sum())
        assert np.array_equal(acc, ref), f"accumulator differs for reference {s_r}"
    dm = ctx.upload_cloud(bottle_5mm)
    hy = ctx.vote(dm, t, dev_crop, 0, 50)
    for h in hy[::3]:
        acc = ctx.vote_debug_accumulator(t, dev_crop, int(h["scene_index"]))
        flat = int(np.argmax(acc))
        assert h["votes"] == acc.reshape(-1)[flat]
        if h["votes"]:
            assert (int(h["model_index"]), int(h["alpha_bin"])) == divmod(flat, acc.shape[1])


def test_c2_full_scene(ctx, bottle, scene_full, dev_bottle, oracle_bottle, table_from_oracle_features):
    """BASELINE config 2 at full size (44 893 reference points): accumulators of sampled reference points
    bit-exact against the oracle, every sampled peak the first maximum of its accumulator, and the
    size-independent property that an interleaved 3-way split of the reference points reproduces the
    single-launch records byte for byte."""
    _, hm = oracle_bottle
    t = table_from_oracle_features
    ds = ctx.upload_cloud(scene_full)
    full = ctx.vote(dev_bottle, t, ds, 0, 1)
    st = ctx.vote_stats()
    assert len(full) == scene_full.shape[0] and np.array_equal(full["scene_index"], np.arange(len(full)))
    assert st["votes"] > 7.0e9 and st["pairs_in_radius"] > 1.4e7
    rng = np.random.default_rng(11)
    for s_r in rng.choice(len(full), 10, replace=False):
        inr, d, a = ctx.vote_debug_pairs(t, ds, int(s_r))
        acc = ctx.vote_debug_accumulator(t, ds, int(s_r))
        ref, votes = hm.vote_accumulate_from_pairs(bottle.shape[0], d[inr > 0], a[inr > 0])
        assert votes == int(acc.sum()) and np.array_equal(acc, ref), f"accumulator differs for reference {s_r}"
        flat = int(np.argmax(acc))
        h = full[int(s_r)]
        assert h["votes"] == acc.reshape(-1)[flat]
        if h["votes"]:
            assert (int(h["model_index"]), int(h["alpha_bin"])) == divmod(flat, acc.shape[1])
    parts = [ctx.vote(dev_bottle, t, ds, g, 3) for g in range(3)]
    merged = np.empty_like(full)
    for g in range(3):
        merged[g::3] = parts[g]
    assert merged.tobytes() == full.tobytes()


def test_k3_dense_scene_flushes_candidate_queue(ctx, bottle, oracle_bottle, table_from_oracle_features):
    """A scene dense enough that one reference point has far more than 2 048 in-radius neighbours: the sweep
    has to flush its candidate queue several times (the barrier-ful branch of phase A)."""
    from yolo_ppf_pose_estimation_b200 import synth
    _, hm = oracle_bottle
    dense = synth.synth_scene(24000, 5).copy()
    c = np.array([0.0, 0.0, 1.5], np.float32)
    dense[:, :3] = (dense[:, :3] - c) * np.float32(0.12) + c   # 2 m scene squeezed into ~25 cm
    ds = ctx.upload_cloud(dense)
    for s_r in (7, 12000):
        inr, d, a = ctx.vote_debug_pairs(table_from_oracle_features, ds, s_r)
        assert inr.sum() > 2 * 2048
        acc = ctx.vote_debug_accumulator(table_from_oracle_features, ds, s_r)
        ref, votes = hm.vote_accumulate_from_pairs(bottle.shape[0], d[inr > 0], a[inr > 0])
        assert votes == int(acc.sum()) and np.array_equal(acc, ref)
    assert ctx.vote_stats()["pairs_in_radius"] == int(inr.sum())


def test_c3_quarter_scale_vs_oracle(ctx, oracle):
    """BASELINE config 3 at quarter scale (2 500-point synthetic model, 25 000-point scene): two accumulator
    slices, buckets of thousands of entries.  Sampled accumulators bit-exact, final pose == oracle's on the
    same hypotheses, and the recovered pose is the scene's ground truth."""
    from yolo_ppf_pose_estimation_b200 import workloads, synth
    wl = workloads.load("c3s")
    feats = oracle.ppf_estimation(wl.model)
    hm = oracle.HashMap(wl.angle_step, wl.dist_step).set_input_feature_cloud(feats)
    dm, ds = ctx.upload_cloud(wl.model), ctx.upload_cloud(wl.scene)
    t = ctx.table_build_from_cloud(dm, wl.angle_step, wl.dist_step)
    assert t.info.n_slices >= 2 and abs(int(t.info.n_entries) - hm.num_entries) <= 4
    tf = ctx.table_build(ctx.features_upload(feats), wl.angle_step, wl.dist_step)
    for s_r in (3, 9999, 20011):
        inr, d, a = ctx.vote_debug_pairs(tf, ds, s_r)
        acc = ctx.vote_debug_accumulator(tf, ds, s_r)
        ref, votes = hm.vote_accumulate_from_pairs(wl.model.shape[0], d[inr > 0], a[inr > 0])
        assert votes == int(acc.sum()) and np.array_equal(acc, ref), s_r
    hy = ctx.vote(dm, tf, ds, 0, 1)
    poses, votes = ctx.cluster(hy, wl.pos_thr, wl.rot_thr)
    rposes, rvotes, _, _ = oracle.cluster(hy, wl.pos_thr, wl.rot_thr)
    assert np.array_equal(votes, rvotes)
    dt, dr = parity.pose_error(poses[0], rposes[0])
    assert dt < 1e-3 and dr < 0.5, (dt, dr)
    dt, da = axis_pose_error(poses[0], synth.gt_pose(2))
    assert dt < 5e-3 and da < 3.0, (dt, da)   # PPF resolution: 1 cm distance step, 12 degree alpha bins


def axis_pose_error(P, G):
    """The synthetic model is a surface of revolution about z: the rotation about its own axis is not
    observable, so compare the translation (the origin lies on the axis) and the axis direction."""
    P, G = np.asarray(P, np.float64), np.asarray(G, np.float64)
    dt = float(np.linalg.norm(P[:3, 3] - G[:3, 3]))
    c = float(np.clip(P[:3, 2] @ G[:3, 2], -1, 1))
    return dt, float(np.degrees(np.arccos(c)))


@pytest.fixture(scope="module")
def c3_full(ctx, oracle):
    """BASELINE config 3 at full size on both sides: the oracle's container for the 10 000-point model (10^8 pairs,
    built sharded over the host cores) and the device table made from the oracle's own signatures (identical floats
    in), seven accumulator slices, the 1024-thread launch shape."""
    from yolo_ppf_pose_estimation_b200 import workloads
    wl = workloads.load("c3")
    th = oracle.host_threads()
    feats = oracle.ppf_estimation(wl.model, n_threads=th)
    hm = oracle.HashMap(wl.angle_step, wl.dist_step).set_input_feature_cloud(feats, n_threads=th)
    dm, ds = ctx.upload_cloud(wl.model), ctx.upload_cloud(wl.scene)
    tf = ctx.table_build(ctx.features_upload(feats), wl.angle_step, wl.dist_step)
    del feats
    hy = ctx.vote(dm, tf, ds, 0, 1)
    st = ctx.vote_stats()
    return wl, hm, dm, ds, tf, hy, st, th


def _c3_sample_refs(wl):
    """one reference point on the object, one on the ground plane, one on a wall, one in a clutter blob"""
    from yolo_ppf_pose_estimation_b200 import synth
    s = wl.scene.astype(np.float64)
    G = synth.gt_pose(2)
    centre = G[:3, 3] + G[:3, :3] @ np.array([0.0, 0.0, 0.09])
    on_object = int(np.argmin(np.linalg.norm(s[:, :3] - centre, axis=1)))
    ground = int(np.flatnonzero((np.abs(s[:, 1] - 0.45) < 0.002) & (s[:, 4] < -0.95) & (np.abs(s[:, 0]) < 0.5))[0])
    wall = int(np.flatnonzero((np.abs(s[:, 2] - 2.5) < 0.002) & (s[:, 5] < -0.95) & (np.abs(s[:, 0]) < 0.5))[0])
    planes = (np.abs(s[:, 1] - 0.45) < 0.01) | (np.abs(s[:, 2] - 2.5) < 0.01) | (np.abs(s[:, 0] + 1.0) < 0.01)
    far = np.linalg.norm(s[:, :3] - centre, axis=1) > 0.3
    clutter = int(np.flatnonzero(~planes & far)[0])
    return {"object": on_object, "ground": ground, "wall": wall, "clutter": clutter}


def test_c3_full_size_vs_oracle(ctx, oracle, c3_full):
    """The headline configuration against the oracle, not against itself: accumulators of reference points on the
    object, on the two kinds of plane and in the clutter bit-exact at seven slices, each hypothesis the first maximum
    of its accumulator with the oracle's pose, the table's bucket statistics those of the oracle's container."""
    wl, hm, dm, ds, tf, hy, st, th = c3_full
    ti = tf.info
    assert ti.n_slices == 7 and ti.phase_cells == 16 and ti.n_alpha == 30
    assert ti.n_entries == hm.num_entries == 99990000 and ti.n_keys == hm.num_keys
    assert 0 < ti.n_merged < ti.n_entries
    assert np.float32(ti.max_dist) == np.float32(hm.model_diameter)
    n = wl.model.shape[0]
    seen = {}
    for what, s_r in _c3_sample_refs(wl).items():
        inr, d, a = ctx.vote_debug_pairs(tf, ds, s_r)
        acc = ctx.vote_debug_accumulator(tf, ds, s_r)
        ref, votes = hm.vote_accumulate_from_pairs(n, d[inr > 0], a[inr > 0], n_threads=th)
        assert votes == int(acc.sum()) == ctx.vote_stats()["votes"], (what, s_r)
        assert np.array_equal(acc, ref), f"accumulator differs for the {what} reference point {s_r}"
        flat = int(np.argmax(acc))
        h = hy[s_r]
        assert h["scene_index"] == s_r and h["votes"] == acc.reshape(-1)[flat]
        assert (int(h["model_index"]), int(h["alpha_bin"])) == divmod(flat, acc.shape[1])
        P = oracle.peak_pose(wl.model, int(h["model_index"]), int(h["alpha_bin"]), wl.scene, s_r, wl.angle_step)
        assert np.abs(P.reshape(-1) - h["pose"]).max() < 2e-5
        seen[what] = (int(inr.sum()), votes)
    print("C3 full size, (in-radius pairs, votes) per sampled reference point:", seen)
    assert seen["object"][1] > 1e8 and seen["ground"][1] > 1e7    # the sample does hit the expensive points


def test_c3_full_size_clustering_vs_oracle(ctx, oracle, c3_full):
    """K4 on all 100 000 hypotheses of config 3 (one cluster of thousands of members on the object: the leader-list
    path): assignments, cluster votes and the three averaged poses against the oracle's greedy loop."""
    wl, hm, dm, ds, tf, hy, st, th = c3_full
    poses, votes = ctx.cluster(hy, wl.pos_thr, wl.rot_thr)
    assign, ncl = ctx.cluster_assignment(len(hy))
    rposes, rvotes, rassign, rncl = oracle.cluster(hy, wl.pos_thr, wl.rot_thr)
    assert ncl == rncl and np.array_equal(assign, rassign)
    assert np.array_equal(votes, rvotes)
    assert np.abs(poses - rposes).max() < 1e-5
    assert np.bincount(rassign).max() > 2000


def test_c3_full_size_properties(ctx, c3_full):
    """Size-independent properties at full size (8.1e12 votes per pass): work counters, the ground-truth pose, and
    reference shards reproducing the single-launch records byte for byte."""
    from yolo_ppf_pose_estimation_b200 import synth
    wl, hm, dm, ds, tf, hy, st, th = c3_full
    # counters of the table made from the oracle's signatures; the table made from the device's own differs by edge pairs
    assert abs(st["votes"] - 8106143691736) < 1e-6 * 8106143691736 and st["pairs_in_radius"] == 99513110
    poses, votes = ctx.cluster(hy, wl.pos_thr, wl.rot_thr)
    dt, da = axis_pose_error(poses[0], synth.gt_pose(2))
    assert dt < 2e-3 and da < 3.0, (dt, da)
    part = ctx.vote(dm, tf, ds, 5, 997)
    assert part.tobytes() == hy[5::997].tobytes()
    # the table built straight from the model cloud (device floats) differs from the oracle's by edge pairs only
    t = ctx.table_build_from_cloud(dm, wl.angle_step, wl.dist_step)
    assert abs(int(t.info.n_entries) - 99990000) <= 64 and t.info.phase_cells == 16
    ctx.vote(dm, t, ds, 0, 997)
    tf_votes = ctx.vote_stats()["votes"]
    ctx.vote(dm, tf, ds, 0, 997)
    assert abs(tf_votes - ctx.vote_stats()["votes"]) < 1e-5 * tf_votes


def test_c4s_library_both_partitionings(ctx, oracle):
    """BASELINE config 4 (eighth-scale scene): the 8-model library against one scene.  Accumulators of sampled
    reference points bit-exact per model; and the two ways of spreading the work over G GPUs — one model per GPU
    (every reference point), or every table on every GPU with the reference points interleaved — give the same
    hypothesis records byte for byte, hence the same poses."""
    from yolo_ppf_pose_estimation_b200 import workloads, synth
    wl = workloads.load("c4s")
    th = oracle.host_threads()
    ds = ctx.upload_cloud(wl.scene)
    rate, n_ref = wl.ref_rate, wl.n_ref
    for k in (0, 3, 7):
        model = wl.models[k]
        feats = oracle.ppf_estimation(model, n_threads=th)
        hm = oracle.HashMap(wl.angle_step, wl.dist_step).set_input_feature_cloud(feats, n_threads=th)
        dm = ctx.upload_cloud(model)
        tf = ctx.table_build(ctx.features_upload(feats), wl.angle_step, wl.dist_step)
        assert tf.info.n_entries == hm.num_entries
        G = synth.library_pose(k, 3)
        centre = G[:3, 3] + G[:3, :3] @ np.array([0.0, 0.0, 0.09])
        near = np.argsort(np.linalg.norm(wl.scene[:, :3].astype(np.float64) - centre, axis=1))[:400]
        on_object = int(near[near % rate == 0][0])      # a reference point of the workload on model k's instance
        for s_r in (on_object, rate * 1234):
            inr, d, a = ctx.vote_debug_pairs(tf, ds, s_r)
            acc = ctx.vote_debug_accumulator(tf, ds, s_r)
            ref, votes = hm.vote_accumulate_from_pairs(model.shape[0], d[inr > 0], a[inr > 0], n_threads=th)
            assert votes == int(acc.sum()) and np.array_equal(acc, ref), (k, s_r)
        # partitioning 1: this model on one GPU, every reference point
        full = ctx.vote(dm, tf, ds, 0, rate, n_ref)
        # partitioning 2: reference points interleaved over 4 ranks, every rank holding this model's table
        merged = np.empty_like(full)
        for r in range(4):
            cnt = (n_ref - r + 3) // 4
            merged[r::4] = ctx.vote(dm, tf, ds, r * rate, 4 * rate, cnt)
        assert merged.tobytes() == full.tobytes()
        poses, votes = ctx.cluster(full, wl.pos_thr, wl.rot_thr)
        rposes, rvotes, _, _ = oracle.cluster(full, wl.pos_thr, wl.rot_thr)
        assert np.array_equal(votes, rvotes) and np.abs(poses - rposes).max() < 1e-5
        # (at an eighth of the scene every 20th point leaves ~100 reference points on an instance: whether the best
        # cluster is the instance is a property of the workload's scale, not of the engine — not asserted here)


@pytest.mark.parametrize("step_deg", [6.0, 14.3239448782706, 25.0])
def test_k3_other_angle_steps(ctx, oracle, bottle, dev_crop, step_deg):
    """6 degrees: 60 phase positions per turn (constant-shift path, 7-bit wrap field); 0.25 rad and
    25 degrees: 2*pi/step is not an integer, every bucket takes the per-entry path (seam band on)."""
    step = np.float32(step_deg) / np.float32(180.0) * np.float32(np.pi)
    feats = oracle.ppf_estimation(bottle)
    hm = oracle.HashMap(step, DIST_STEP).set_input_feature_cloud(feats)
    t = ctx.table_build(ctx.features_upload(feats), step, DIST_STEP)
    assert t.info.n_entries == hm.num_entries
    assert (t.info.phase_cells > 1) == (step_deg == 6.0)
    for s_r in (5, 600):
        inr, d, a = ctx.vote_debug_pairs(t, dev_crop, s_r)
        acc = ctx.vote_debug_accumulator(t, dev_crop, s_r)
        ref, votes = hm.vote_accumulate_from_pairs(bottle.shape[0], d[inr > 0], a[inr > 0])
        assert votes == int(acc.sum())
        assert np.array_equal(acc, ref), f"accumulator differs for reference {s_r}"


def test_k3_peer_scatter_epilogue(ctx, dev_bottle, dev_crop, table_fused):
    """The multi-GPU exchange fused into the vote epilogue: two "ranks" (here two calls on one GPU) write their
    interleaved shares into BOTH record buffers; each buffer then equals the single-launch result."""
    full = ctx.vote(dev_bottle, table_fused, dev_crop, 0, 1)
    n = len(full)
    bufs = [ctx.hyp_buffer_create(n)[0] for _ in range(2)]
    for rank in range(2):
        count = (n - rank + 1) // 2
        ctx.vote_scatter_device(dev_bottle, table_fused, dev_crop, rank, 2, count, bufs, rank, 2)
    for b in bufs:
        got = ctx.download_hypotheses(b, n)
        assert got.tobytes() == full.tobytes()
        ctx.hyp_buffer_release(b, False)
    from yolo_ppf_pose_estimation_b200 import capi
    with pytest.raises(capi.B200PPFError):
        ctx.vote_scatter_device(dev_bottle, table_fused, dev_crop, 0, 1, n, [], 0, 1)


def test_multi_gpu_group_in_one_process(ctx, bottle, scene_crop, dev_bottle, dev_crop, table_fused):
    """b200ppf_multi_*: the group machinery (interleaved shares, records stored into every rank's buffer by the vote
    epilogue, device-side flags, the waiting kernel) with three 'ranks' that are three contexts on this one GPU:
    the poses are those of the single-context align, step after step (the two buffer sets alternate)."""
    from yolo_ppf_pose_estimation_b200 import capi
    final, poses, votes = ctx.register(dev_bottle, table_fused, dev_crop, ref_rate=5)
    m = capi.Multi([0, 0, 0])
    assert m.size == 3
    m.train(bottle, ANGLE_STEP, DIST_STEP)
    m.scene(scene_crop)
    for _ in range(3):
        f2, p2, v2 = m.register(ref_rate=5)
        assert np.array_equal(v2, votes) and np.array_equal(p2, poses) and np.array_equal(f2, final)
    # another scene size on the same handle (buffers are re-made when they are too small), every point a reference
    f1, p1, v1 = ctx.register(dev_bottle, table_fused, dev_crop, ref_rate=1)
    f3, p3, v3 = m.register(ref_rate=1)
    assert np.array_equal(v3, v1) and np.array_equal(p3, p1)
    with pytest.raises(capi.B200PPFError):
        capi.Multi([0, 99])
    m.close()


def test_multi_gpu_group_across_processes(tmp_path, ctx, dev_bottle, dev_crop, table_fused):
    """b200ppf_group_*: two processes (both on this GPU), buffers mapped into one another through the CUDA IPC handle
    blobs, exchanged here through files: both ranks return the single-context poses."""
    final, poses, votes = ctx.register(dev_bottle, table_fused, dev_crop, ref_rate=5)
    code = f"""
import sys, os, time, numpy as np
sys.path.insert(0, {ROOT!r}); sys.path.insert(0, {os.path.join(ROOT, 'tests')!r})
from yolo_ppf_pose_estimation_b200 import capi
from conftest import ANGLE_STEP, DIST_STEP, load_cloud
rank, world, d = int(sys.argv[1]), 2, sys.argv[2]
m, s = load_cloud('bottle_1cm'), load_cloud('scene_crop_1cm')
c = capi.Context(0)
dm, ds = c.upload_cloud(m), c.upload_cloud(s)
t = c.table_build_from_cloud(dm, ANGLE_STEP, DIST_STEP)
g = capi.Group(c, rank, world, (s.shape[0] + 4) // 5 + 8)
np.save(os.path.join(d, f'h{{rank}}.tmp.npy'), g.handles); os.replace(os.path.join(d, f'h{{rank}}.tmp.npy'), os.path.join(d, f'h{{rank}}.npy'))
hs = []
for r in range(world):
    p = os.path.join(d, f'h{{r}}.npy')
    for _ in range(600):
        if os.path.exists(p): break
        time.sleep(0.05)
    hs.append(np.load(p))
g.connect(hs)
for step in range(3):
    poses, votes = g.register(dm, t, ds, 5)
np.savez(os.path.join(d, f'out{{rank}}.npz'), poses=poses, votes=votes)
open(os.path.join(d, f'done{{rank}}'), 'w').close()
for r in range(world):          # keep the buffers mapped until the peer is done with them
    for _ in range(600):
        if os.path.exists(os.path.join(d, f'done{{r}}')): break
        time.sleep(0.05)
g.close()
print('RANK_OK')
"""
    procs = [subprocess.Popen([sys.executable, "-c", code, str(r), str(tmp_path)], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
             for r in range(2)]
    outs = [p.communicate(timeout=300)[0] for p in procs]
    for r, o in enumerate(outs):
        assert "RANK_OK" in o, o
        z = np.load(tmp_path / f"out{r}.npz")
        assert np.array_equal(z["votes"], votes) and np.array_equal(z["poses"], poses)


def test_k3_alpha_bins_on_device(ctx):
    from yolo_ppf_pose_estimation_b200 import capi
    rng = np.random.default_rng(5)
    am = rng.uniform(-np.pi, np.pi, 1 << 20).astype(np.float32)
    as_ = rng.uniform(-np.pi, np.pi, 1 << 20).astype(np.float32)
    for step in (ANGLE_STEP, np.float32(0.25), np.float32(np.pi / 180)):
        for mode in (0, 1):
            fd, ed = capi.debug_alpha_bins(am, as_, step, mode, ctx)
            fh, eh = capi.debug_alpha_bins(am, as_, step, mode, None)
            assert np.array_equal(fd, ed) and np.array_equal(ed, eh) and np.array_equal(fh, eh)


def test_k3_alpha_mode_b(bottle, scene_crop, oracle, oracle_bottle):
    from yolo_ppf_pose_estimation_b200 import capi
    feats, hm = oracle_bottle
    c = capi.Context(0, alpha_mode=capi.ALPHA_MODE_B)
    t = c.table_build(c.features_upload(feats), ANGLE_STEP, DIST_STEP)
    ds = c.upload_cloud(scene_crop)
    for s_r in (5, 600):
        inr, d, a = c.vote_debug_pairs(t, ds, s_r)
        acc = c.vote_debug_accumulator(t, ds, s_r)
        ref, _ = hm.vote_accumulate_from_pairs(bottle.shape[0], d[inr > 0], a[inr > 0], alpha_mode=oracle.ALPHA_MODE_B)
        assert np.array_equal(acc, ref)


# ---- K4 / K5 / align ------------------------------------------------------------------------------

def test_k4_cluster_vs_oracle(ctx, bottle, scene_crop, oracle, oracle_bottle):
    _, hm = oracle_bottle
    hyps, _ = hm.vote(bottle, scene_crop, 0, 1, n_threads=oracle.max_threads())
    for pos_thr, rot_thr in ((0.01, 20 / 180 * np.pi), (0.006, 12 / 180 * np.pi), (0.2, 30 / 180 * np.pi)):
        poses, votes = ctx.cluster(hyps, pos_thr, rot_thr)
        rposes, rvotes, rassign, rncl = oracle.cluster(hyps, pos_thr, rot_thr)
        assign, ncl = ctx.cluster_assignment(len(hyps))
        assert ncl == rncl
        assert np.array_equal(assign, rassign)
        assert np.array_equal(votes, rvotes)
        assert np.abs(poses - rposes).max() < 1e-5


def test_k4_small_and_degenerate(ctx, oracle):
    from yolo_ppf_pose_estimation_b200.capi import HYP_DTYPE
    h = np.zeros(1, HYP_DTYPE)
    h["pose"][0] = np.eye(4, dtype=np.float32)[:3].reshape(-1)
    h["votes"] = 7
    poses, votes = ctx.cluster(h)
    assert len(poses) == 1 and votes[0] == 7 and np.allclose(poses[0], np.eye(4), atol=1e-6)
    # all-identical poses collapse into one cluster with summed votes
    h = np.repeat(h, 2500)
    h["votes"] = np.arange(2500) % 11
    h["scene_index"] = np.arange(2500)
    poses, votes = ctx.cluster(h)
    rp, rv, ra, rn = oracle.cluster(h)
    assert len(poses) == 1 and votes[0] == h["votes"].sum() == rv[0]
    poses, votes = ctx.cluster(h[:0])
    assert len(poses) == 0


def test_k5_transform(ctx, bottle, dev_bottle, oracle):
    M = np.eye(4, dtype=np.float32)
    M[:3, :3] = np.array([[0, -1, 0], [1, 0, 0], [0, 0, 1]], np.float32)
    M[:3, 3] = (0.1, -0.2, 0.3)
    out = ctx.transform(dev_bottle, M)
    assert np.array_equal(out, oracle.transform(bottle, M))


def test_align_final_pose_vs_oracle(ctx, bottle, scene_crop, dev_bottle, dev_crop, oracle, oracle_bottle, table_fused):
    """PPFRegistration::align end to end, device floats throughout: final pose within 1 mm / 0.5 deg."""
    _, hm = oracle_bottle
    final, poses, votes = ctx.register(dev_bottle, table_fused, dev_crop, ref_rate=5)
    rfinal, rposes, rvotes, _ = hm.register(bottle, scene_crop, ref_rate=5, n_threads=oracle.max_threads())
    dt, dr = parity.pose_error(final, rfinal)
    assert dt < parity.POSE_T_TOL and dr < parity.POSE_R_TOL_DEG, (dt, dr)
    assert len(poses) == len(rposes)
    assert np.abs(votes.astype(np.int64) - rvotes.astype(np.int64)).max() <= 0.02 * rvotes.max() + 3


def test_align_recovers_known_pose(ctx, bottle, dev_bottle, table_fused):
    """Model matched against a rigidly moved copy of itself returns the motion (GT known exactly)."""
    from scipy.spatial.transform import Rotation as Rot
    R = Rot.from_rotvec([0.3, -0.5, 0.8]).as_matrix()
    t = np.array([0.1, -0.05, 0.3])
    s = bottle.astype(np.float64).copy()
    s[:, :3] = s[:, :3] @ R.T + t
    s[:, 3:] = s[:, 3:] @ R.T
    final, _, _ = ctx.register(dev_bottle, table_fused, ctx.upload_cloud(s.astype(np.float32)), ref_rate=5)
    G = np.eye(4)
    G[:3, :3], G[:3, 3] = R, t
    dt, dr = parity.pose_error(final, G)
    assert dt < 3e-3 and dr < 1.0, (dt, dr)


# ---- edge cases and errors ----------------------------------------------------------------------------

def test_errors_and_edges(ctx, bottle, dev_bottle, dev_crop, table_fused):
    from yolo_ppf_pose_estimation_b200.capi import B200PPFError
    with pytest.raises(B200PPFError):  # reference range beyond the scene
        ctx.vote(dev_bottle, table_fused, dev_crop, 0, 1, dev_crop.size + 1)
    with pytest.raises(B200PPFError):  # model / table mismatch
        ctx.vote(dev_crop, table_fused, dev_crop, 0, 1, 1)
    with pytest.raises(B200PPFError):  # not n*n signatures
        ctx.table_build(ctx.features_upload(np.zeros((10, 5), np.float32)), ANGLE_STEP, DIST_STEP)
    with pytest.raises(B200PPFError):
        ctx.table_build_from_cloud(dev_bottle, 0.0, DIST_STEP)
    with pytest.raises(B200PPFError):  # discretisation too fine for 32-bit packed keys
        ctx.table_build_from_cloud(dev_bottle, 1e-4, 1e-6)
    # NaN points are dropped at upload
    c = bottle[:50].copy()
    c[3, 0] = np.nan
    c[10, 4] = np.nan
    assert ctx.upload_cloud(c).size == 48
    # PointNormal layout (stride 12, normals at 4) == N x 6 layout
    pn = np.zeros((bottle.shape[0], 12), np.float32)
    pn[:, :3], pn[:, 3], pn[:, 4:7] = bottle[:, :3], 1.0, bottle[:, 3:]
    a = ctx.vote(ctx.upload_cloud(pn), table_fused, dev_crop, 0, 50)
    b = ctx.vote(dev_bottle, table_fused, dev_crop, 0, 50)
    assert a.tobytes() == b.tobytes()
    # duplicate points and a 2-point model: invalid pairs are skipped, nothing crashes
    dup = np.concatenate([bottle[:40], bottle[:3]])
    t = ctx.table_build_from_cloud(ctx.upload_cloud(dup), ANGLE_STEP, DIST_STEP)
    assert t.info.n_entries <= 43 * 42 - 6
    t2 = ctx.table_build_from_cloud(ctx.upload_cloud(bottle[:2]), ANGLE_STEP, DIST_STEP)
    assert t2.info.n_entries <= 2
    # a scene far away from everything: zero votes, hypotheses still emitted (PCL pushes one per reference)
    far = bottle[:30].copy()
    far[:, :3] = far[:, :3] * 100.0
    hy = ctx.vote(dev_bottle, table_fused, ctx.upload_cloud(far), 0, 1)
    assert len(hy) == 30 and (hy["votes"] == 0).all() and (hy["model_index"] == 0).all()


# ---- the PCL-shaped C++ surface ------------------------------------------------------------------------

def _icp_case(n_model=20000, n_scene=40000):
    """Model, YOLO-crop-like scene around the instance, ground truth and five perturbed start poses."""
    from yolo_ppf_pose_estimation_b200 import synth
    model = synth.synth_model(n_model, 1)
    G = synth.gt_pose(2)
    sc = synth.synth_scene(n_scene, 2, model_seed=1)
    centre = G[:3, 3] + G[:3, :3] @ np.array([0.0, 0.0, 0.09])
    scene = sc[np.linalg.norm(sc[:, :3] - centre, axis=1) < 0.25]
    starts = []
    for k, (ang, tr) in enumerate(((0.03, 0.003), (0.1, 0.01), (0.2, 0.02), (0.05, 0.03), (0.0, 0.0))):
        axis = np.array([0.3, 1.0, 0.2 + 0.3 * k])
        axis /= np.linalg.norm(axis)
        K = np.array([[0, -axis[2], axis[1]], [axis[2], 0, -axis[0]], [-axis[1], axis[0], 0]])
        D = np.eye(4)
        D[:3, :3] = np.eye(3) + np.sin(ang) * K + (1 - np.cos(ang)) * K @ K
        D[:3, 3] = (tr, -tr, 0.5 * tr)
        C, Ci = np.eye(4), np.eye(4)
        C[:3, 3], Ci[:3, 3] = centre, -centre
        starts.append(C @ D @ Ci @ G)
    return model, scene, G, np.array(starts)


def test_k6_icp_vs_oracle(ctx, oracle):
    """The reference's ICP(100, 0.005, 2.5, 8).registerModelToScene on five start poses at once: same
    iteration count and poses as the oracle (double reductions differ in order only), and the scene's ground
    truth recovered to the noise level."""
    model, scene, G, starts = _icp_case()
    dm, ds = ctx.upload_cloud(model), ctx.upload_cloud(scene)
    P, res, it = ctx.icp_refine(dm, ds, starts)
    R, rres, rit = oracle.icp_refine(model, scene, starts)
    assert abs(it - rit) <= 2, (it, rit)
    for k in range(len(starts)):
        dt, dr = parity.pose_error(P[k], R[k])
        assert dt < 2e-5 and dr < 0.005, (k, dt, dr)          # 20 um / 0.005 degrees between GPU and oracle
        assert abs(res[k] - rres[k]) <= 1e-6 * max(1.0, rres[k])
        dt, da = axis_pose_error(P[k], G)
        assert dt < 5e-4 and da < 0.3, (k, dt, da)            # 0.5 mm sensor noise in the scene
    assert ctx.timings()["icp_ms"] > 0
    # fewer levels / no rejection / one pose: the parameters reach the kernel
    P1, _, it1 = ctx.icp_refine(dm, ds, starts[:1], max_iterations=10, rejection_scale=0.0, num_levels=3)
    R1, _, rit1 = oracle.icp_refine(model, scene, starts[:1], max_iterations=10, rejection_scale=0.0, num_levels=3)
    assert it1 == rit1 and parity.pose_error(P1[0], R1[0])[0] < 2e-5
    # a thinner model (2 500 points): the coarsest levels hold ~20 samples; still the same trajectory
    thin = model[::8]
    Ps, _, its = ctx.icp_refine(ctx.upload_cloud(thin), ds, starts[:2])
    Rs, _, rits = oracle.icp_refine(thin, scene, starts[:2])
    assert abs(its - rits) <= 2
    for k in range(2):
        dt, dr = parity.pose_error(Ps[k], Rs[k])
        assert dt < 1e-4 and dr < 0.02, (k, dt, dr)


def test_k6_icp_on_the_reference_object(ctx, oracle, oracle_bottle, bottle, scene_crop, dev_bottle, dev_crop):
    """The reference's own sizes (543-point model, 934-point crop, 8 levels: 4 samples at the coarsest, fewer correspondences
    than unknowns): the minimum-norm solve keeps both sides on the same trajectory where the elimination of round 1 let
    them fly apart (metres) — device and oracle end at the same pose, near the PPF pose they started from."""
    _, hm = oracle_bottle
    _, poses, votes, _ = hm.register(bottle, scene_crop, ref_rate=5, n_threads=4)
    starts = poses[:3].astype(np.float64)
    P, res, it = ctx.icp_refine(dev_bottle, dev_crop, starts)
    R, rres, rit = oracle.icp_refine(bottle, scene_crop, starts)
    c = np.append(bottle[:, :3].mean(axis=0).astype(np.float64), 1.0)
    assert (res < 1.0).all() and (rres < 1.0).all()                      # no 1e10 sentinel on either side
    assert np.linalg.norm((R[0] @ c - starts[0] @ c)[:3]) < 0.02        # the best pose stays on the object
    for k in range(len(starts)):
        moved = np.linalg.norm((P[k] @ c - R[k] @ c)[:3])
        assert moved < 1e-3 and abs(res[k] - rres[k]) <= 1e-3 * max(1.0, rres[k]), (k, moved, res[k], rres[k])


def test_cpp_pcl_shim_end_to_end(tmp_path, ctx, bottle, scene_crop, dev_bottle, dev_crop, oracle_bottle):
    """tests/cpp/pcl_shim_example.cpp — PPFEstimation::compute -> PPFHashMapSearch::setInputFeatureCloud
    -> PPFRegistration::align through include/pcl_compat — gives the C-ABI result."""
    from yolo_ppf_pose_estimation_b200 import build
    lib = build.build()
    bottle.astype(np.float32).tofile(tmp_path / "bottle_1cm.f32")
    scene_crop.astype(np.float32).tofile(tmp_path / "scene_crop_1cm.f32")
    exe = tmp_path / "pcl_shim_example"
    cmd = ["/usr/bin/g++", "-std=c++14", "-O1", "-I", os.path.join(ROOT, "include", "pcl_compat"), "-I",
           os.path.join(ROOT, "include"), os.path.join(ROOT, "tests", "cpp", "pcl_shim_example.cpp"), "-o", str(exe),
           "-L", os.path.dirname(lib), "-lb200ppf", f"-Wl,-rpath,{os.path.dirname(lib)}"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    r = subprocess.run([str(exe), str(tmp_path)], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    lines = r.stdout.strip().splitlines()
    M = np.array([[float(x) for x in ln.split()] for ln in lines[:4]], np.float32)
    # the same pipeline through the C ABI: two-step table from the device's own signatures
    t = ctx.table_build(ctx.features_compute(dev_bottle), ANGLE_STEP, DIST_STEP)
    final, poses, votes = ctx.register(dev_bottle, t, dev_crop, ref_rate=5)
    assert np.array_equal(M, final)
    _, hm = oracle_bottle
    info = dict(zip(lines[4].split()[::2], lines[4].split()[1::2]))
    assert np.float32(info["model_diameter"]) == np.float32(hm.model_diameter)
    assert int(info["features"]) == 543 * 543 and int(info["output"]) == 543 and int(info["candidates"]) == len(poses)
    out0 = np.array([float(x) for x in lines[6].split()[1:]], np.float32)
    assert np.array_equal(out0, ctx.transform(dev_bottle, final)[0])
    bucket = lines[5].split()
    assert int(bucket[1]) >= 1 and (int(bucket[3]), int(bucket[4])) <= (0, 1)
    assert lines[7].split() == ["reloaded_table_same_pose", "1"]
    assert lines[8].split() == ["copied_table_same_answers", "1"]  # PPFHashMapSearch::makeShared()
    # the same binary with B200PPF_DEVICES=0,0: PPFRegistration::align goes through b200ppf_multi_* (two contexts on
    # this GPU stand in for two GPUs) — same table copied device to device, same poses, same output
    r2 = subprocess.run([str(exe), str(tmp_path)], capture_output=True, text=True, timeout=300,
                        env=dict(os.environ, B200PPF_DEVICES="0,0"))
    assert r2.returncode == 0, r2.stdout + r2.stderr
    assert r2.stdout.strip().splitlines()[:9] == lines[:9]


def test_bench_dump_outputs_are_the_align_result(tmp_path, ctx, dev_bottle, dev_crop, table_fused):
    """bench.py --dump-outputs on c1 (the 1 cm bottle against the crop, every 5th scene point a reference): the poses and
    votes of its last timed step are those b200ppf_register returns on the same clouds, and those its JSON line reports."""
    import json
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "c1", "--steps", "2", "--warmup", "3",
                        "--no-cpu", "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=600,
                       env=dict(os.environ, BENCH_CLOCKS="0"))
    assert r.returncode == 0, r.stderr
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["steps"] == 2
    _, poses, votes = ctx.register(dev_bottle, table_fused, dev_crop, ref_rate=5)
    dumped_poses, dumped_votes = np.load(tmp_path / "poses.npy"), np.load(tmp_path / "votes.npy")
    assert len(votes) > 0 and np.array_equal(dumped_poses, poses) and np.array_equal(dumped_votes, votes.astype(np.float64))
    assert line["result"]["votes"] == [int(v) for v in dumped_votes]
