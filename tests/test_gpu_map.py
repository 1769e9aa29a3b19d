"""GPU parity of the corrected global map (fast_lio_sam_qn.cpp:302-316, :398-411, :435-449): every keyframe transformed by
its corrected pose, merged in keyframe order, one pcl::VoxelGrid -- bit-identical to the oracle's transform_pcd + voxelize."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def seq(synth):
    return synth.make_sequence(7, 140, pts_per_keyframe=6000, spacing=3.0)


def _store(ctx, seq, poses=None):
    kf = ctx.keyframes()
    for c, T, t in zip(seq["clouds"], seq["poses"] if poses is None else poses, seq["stamps"]):
        kf.add(c, T, t)
    return kf


@pytest.fixture(scope="module")
def store(ctx, seq):
    kf = _store(ctx, seq)
    yield kf
    kf.destroy()


def _merged(oracle, seq, n, poses=None):
    poses = seq["poses"] if poses is None else poses
    return np.concatenate([oracle.transform_pcd(seq["clouds"][i], poses[i]) for i in range(n)])


def _key_bits(merged, leaf):
    """ceil(log2(dx * dy * dz)) of pcl::VoxelGrid's grid over the merged cloud (fp32, as the kernels compute it)."""
    inv = np.float32(1.0) / np.float32(leaf)
    lo, hi = merged[:, :3].min(0), merged[:, :3].max(0)
    div = np.floor(hi * inv).astype(np.int64) - np.floor(lo * inv).astype(np.int64) + 1
    return int(np.ceil(np.log2(float(np.prod(div)))))


@pytest.mark.parametrize("n_keyframes", [0, 1, 57, 140])
def test_map_equals_oracle(store, oracle, seq, n_keyframes):
    got, voxelized = store.build_map(0.3, n_keyframes)
    want = oracle.voxelize(_merged(oracle, seq, n_keyframes or len(seq["clouds"])), 0.3)
    assert voxelized
    assert np.array_equal(got, want)  # same count, same order, same bits, intensity included


def test_both_sort_paths(store, oracle, seq):
    """0.3 m: a 24-bit grid, sorted with 8-bit digits; 0.1 m: 28 bits, the 11-bit digits of the sub-map grid."""
    merged = _merged(oracle, seq, len(seq["clouds"]))
    assert _key_bits(merged, 0.3) <= 24 < _key_bits(merged, 0.1)
    for leaf in (0.3, 0.1):
        got, voxelized = store.build_map(leaf)
        assert voxelized and np.array_equal(got, oracle.voxelize(merged, leaf)), leaf


def test_overflow_guard_returns_merged_cloud(store, oracle, seq):
    got, voxelized = store.build_map(0.01)
    assert not voxelized
    assert np.array_equal(got, _merged(oracle, seq, len(seq["clouds"])))


def test_corrected_poses_are_used(ctx, oracle, seq):
    kf = _store(ctx, seq)
    try:
        before, _ = kf.build_map(0.3)
        for i, T in enumerate(seq["true_poses"]):
            kf.set_pose(i, T)
        after, _ = kf.build_map(0.3)
    finally:
        kf.destroy()
    want = oracle.voxelize(_merged(oracle, seq, len(seq["clouds"]), seq["true_poses"]), 0.3)
    assert np.array_equal(after, want)
    assert before.shape != after.shape or not np.array_equal(before, after)


def test_map_of_one_keyframe_equals_assembled_cloud(ctx, store):
    """The two device paths agree: the map of keyframe 0 is assemble()'s Quatro-mode source cloud of keyframe 0."""
    import b200reg
    got, _ = store.build_map(0.3, 1)
    cfg = b200reg.default_loop_config()
    cfg.enable_quatro, cfg.enable_submap_matching = 1, 0
    (sc,), (dc,) = store.assemble([0], [0], cfg, n_keyframes=1)
    try:
        assert np.array_equal(ctx.cloud_points(sc), got[:, :3])
    finally:
        sc.destroy()
        dc.destroy()


def test_map_at_scale(ctx, oracle, synth):
    """18 M points: thousands of tiles in every kernel, 9k blocks in the transform."""
    big = synth.make_sequence(5, 600, pts_per_keyframe=30000, threads=8)
    kf = ctx.keyframes()
    try:
        kf.reserve(600 * 30000)
        for c, T, t in zip(big["clouds"], big["poses"], big["stamps"]):
            kf.add(c, T, t)
        got, voxelized = kf.build_map(0.3)
    finally:
        kf.destroy()
    want = oracle.voxelize(_merged(oracle, big, 600), 0.3)
    assert voxelized and len(want) > 200000
    assert np.array_equal(got, want)


def test_map_is_deterministic_and_leaves_loop_closure_alone(store):
    q = np.array([137, 139, 118], np.int32)
    closest = store.fetch_closest(q)
    before, _ = store.perform_loop_closure(q, closest)
    a, _ = store.build_map(0.3)
    b, _ = store.build_map(0.3)
    assert a.tobytes() == b.tobytes()
    after, _ = store.perform_loop_closure(q, closest)
    for x, y in zip(before, after):
        assert np.array_equal(x["T"], y["T"]) and x["fitness"] == y["fitness"] and x["valid"] == y["valid"]


def test_map_argument_errors(ctx, store):
    import b200reg
    empty = ctx.keyframes()
    try:
        with pytest.raises(b200reg.B200RegError):
            empty.build_map(0.3)
    finally:
        empty.destroy()
    for nk in (-1, 141):
        with pytest.raises(b200reg.B200RegError):
            store.build_map(0.3, nk)
    for leaf in (0.0, -0.3):
        with pytest.raises(b200reg.B200RegError):
            store.build_map(leaf)
