"""GPU parity tests for the Nano-GICP half of the path: CUDA (through the C ABI) vs the CPU oracle.

Bars (BASELINE.json north_star): k-NN / correspondence indices bit-exact, squared distances
bit-exact (fp32), final SE(3) within 1e-4 rad / 1e-3 m of the oracle.
"""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROT_TOL = 1e-4   # rad
TRANS_TOL = 1e-3  # m


def _tie_ok(idx_g, d2_g, idx_o, d2_o):
    """Indices must match except inside runs of exactly equal d2 (SURVEY App. A.3)."""
    assert np.array_equal(d2_g, d2_o), "squared distances differ"
    bad = idx_g != idx_o
    if not bad.any():
        return
    # a mismatch is only legal where the neighbouring slot holds the same d2
    rows, cols = np.nonzero(bad)
    for r, c in zip(rows, cols):
        same = (c > 0 and d2_o[r, c - 1] == d2_o[r, c]) or (c + 1 < d2_o.shape[1] and d2_o[r, c + 1] == d2_o[r, c])
        assert same, "index mismatch without a distance tie at query %d slot %d" % (r, c)


def test_knn15_self_queries_exact(ctx, oracle, pair20k):
    src, dst, _ = pair20k
    cl, = ctx.create_clouds([dst])
    idx, d2 = ctx.knn(cl, dst, 15)
    oidx, od2 = oracle.knn(dst, dst, 15)
    assert np.array_equal(d2, od2)
    assert np.array_equal(idx, oidx)
    assert (np.diff(d2, axis=1) >= 0).all()
    assert np.array_equal(idx[:, 0], np.arange(len(dst)))  # continuous noise: every point is its own 1-NN
    cl.destroy()


def test_knn_against_reference_nanoflann(ctx, pair20k):
    """The reference kd-tree's answers on seeded samples of these query sets: golden/knn_ref_nanoflann_20k.npz."""
    import os
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "knn_ref_nanoflann_20k.npz"))
    src, dst, _ = pair20k
    cl, = ctx.create_clouds([dst])
    for name, k, q in (("src1", 1, src), ("self15", 15, dst[:8000]), ("shift1", 1, src + np.float32(3.0)), ("src20", 20, src[:4000])):
        gi, gd = ctx.knn(cl, q[g["rows_" + name]], k)
        _tie_ok(gi, gd, g["idx_" + name], g["d2_" + name])
    cl.destroy()


def test_knn1_far_queries_exact(ctx, oracle, pair20k):
    src, dst, _ = pair20k
    cl, = ctx.create_clouds([dst])
    rng = np.random.default_rng(5)
    q = (src[:, :3] + rng.normal(0, 4.0, (len(src), 3))).astype(np.float32)
    q[:50] *= 30.0  # far outside the cloud's bounding box
    gi, gd = ctx.knn(cl, q, 1)
    oi, od = oracle.knn(dst, q, 1)
    assert np.array_equal(gd, od) and np.array_equal(gi, oi)
    cl.destroy()


def test_knn_small_and_ragged_clouds(ctx, oracle):
    rng = np.random.default_rng(11)
    for n in (1, 7, 8, 9, 17, 63, 64, 65, 1000):
        pts = rng.normal(0, 5, (n, 4)).astype(np.float32)
        q = rng.normal(0, 6, (33, 3)).astype(np.float32)
        cl, = ctx.create_clouds([pts])
        for k in (1, 15):
            gi, gd = ctx.knn(cl, q, k)
            oi, od = oracle.knn(pts, q, k, brute=True)
            kk = min(k, n)
            assert np.array_equal(gi[:, :kk], oi[:, :kk]) and np.array_equal(gd[:, :kk], od[:, :kk])
            assert (gi[:, kk:] == -1).all()
        cl.destroy()


def test_knn_duplicate_points_tie_rule(ctx, oracle):
    """Exact duplicates: ties must resolve to the lower original index (SURVEY App. A.3)."""
    rng = np.random.default_rng(3)
    base = rng.normal(0, 3, (500, 3)).astype(np.float32)
    pts = np.concatenate([base, base, base])[rng.permutation(1500)]
    cl, = ctx.create_clouds([pts])
    gi, gd = ctx.knn(cl, base, 15)
    oi, od = oracle.knn(pts, base, 15, brute=True)
    assert np.array_equal(gd, od) and np.array_equal(gi, oi)
    cl.destroy()


def test_covariances_match_oracle(ctx, oracle, pair20k):
    src, dst, _ = pair20k
    cl, = ctx.create_clouds([dst])
    ctx.covariances([cl], 15)
    g = ctx.get_covariances(cl)
    o = oracle.covariances(dst, 15)
    err = np.abs(g - o).reshape(len(dst), -1).max(1)
    # plane normals are ill-conditioned where the two smallest eigenvalues coincide (edges, poles);
    # the bulk must agree to fp64 round-off and no point may be wildly off.
    assert np.median(err) < 1e-12
    assert np.quantile(err, 0.999) < 1e-6
    # structure: symmetric, eigenvalues (1, 1, 1e-3)
    assert np.allclose(g, np.swapaxes(g, 1, 2), atol=0)
    ev = np.linalg.eigvalsh(g[::97])
    assert np.allclose(ev, [1e-3, 1.0, 1.0], atol=1e-9)
    cl.destroy()


def test_linearize_matches_oracle(ctx, oracle, synth, pair20k):
    src, dst, _ = pair20k
    cs, ct = ctx.create_clouds([src, dst])
    ctx.covariances([cs, ct], 15)
    cov_s, cov_t = ctx.get_covariances(cs), ctx.get_covariances(ct)
    for T in (np.eye(4), synth.se3(yaw=0.02, pitch=-0.004, t=(0.3, -0.2, 0.05))):
        g = ctx.linearize(cs, ct, T)
        o = oracle.linearize(src, dst, cov_s, cov_t, T)  # same covariances in: isolates the linearize pass
        assert np.array_equal(g["corr"], o["corr"]), "correspondence indices must be bit-exact"
        assert np.array_equal(g["sqd"], o["sqd"])
        scale = np.abs(o["H"]).max()
        assert np.abs(g["H"] - o["H"]).max() < 1e-9 * scale
        assert np.abs(g["b"] - o["b"]).max() < 1e-9 * max(np.abs(o["b"]).max(), 1.0)
        assert abs(g["err"] - o["err"]) < 1e-9 * abs(o["err"])
    # tight correspondence gate: rejected points must be -1 on both sides
    g = ctx.linearize(cs, ct, np.eye(4), max_corr_dist=0.25)
    o = oracle.linearize(src, dst, cov_s, cov_t, np.eye(4), max_corr_dist=0.25)
    assert (o["corr"] < 0).any() and np.array_equal(g["corr"], o["corr"])
    assert np.abs(g["H"] - o["H"]).max() < 1e-9 * np.abs(o["H"]).max()
    cs.destroy(); ct.destroy()


def _check_pair(ctx, oracle, synth, src, dst, Texp=None):
    g = ctx.icp_alignment([src], [dst])[0]
    o = oracle.gicp_align(src, dst)
    rot, trans = synth.se3_error(g["T"], o["T"])
    assert rot < ROT_TOL and trans < TRANS_TOL, (rot, trans)
    assert g["converged"] == o["converged"]
    assert g["n_linearize"] == o["n_linearize"] and g["n_error"] == o["n_error"]
    assert g["iterations"] == o["iterations"]
    assert abs(g["fitness"] - o["fitness"]) < 1e-5 * max(o["fitness"], 1e-3)
    assert np.allclose(g["Tf"], g["T"].astype(np.float32), atol=0)
    if Texp is not None:
        rot, trans = synth.se3_error(g["T"], Texp)
        assert rot < 5e-3 and trans < 5e-2, ("ground truth", rot, trans)
    return g, o


def test_gicp_align_matches_oracle_20k(ctx, oracle, synth, pair20k):
    src, dst, Texp = pair20k
    _check_pair(ctx, oracle, synth, src, dst, Texp)


def test_gicp_align_ragged_sizes(ctx, oracle, synth, pair5k):
    src, dst, Texp = pair5k
    _check_pair(ctx, oracle, synth, src, dst, Texp)


def test_gicp_align_pointxyzi_stride(ctx, oracle, synth, pair5k):
    """pcl::PointXYZI records (32 B stride) upload without repacking."""
    src, dst, _ = pair5k

    def xyzi32(a):
        out = np.zeros((len(a), 8), np.float32)
        out[:, :3] = a[:, :3]
        out[:, 3] = 1.0
        out[:, 4] = a[:, 3]
        return out
    g8 = ctx.icp_alignment([xyzi32(src)], [xyzi32(dst)])[0]
    g4 = ctx.icp_alignment([src], [dst])[0]
    assert np.array_equal(g8["T"], g4["T"]) and g8["fitness"] == g4["fitness"]


def test_batch_equals_single_and_is_deterministic(ctx, oracle, synth):
    pairs = [synth.make_pair(1100 + i, 4000 + 500 * i, 5000 - 300 * i) for i in range(5)]
    srcs = [p[0] for p in pairs]
    dsts = [p[1] for p in pairs]
    batch = ctx.icp_alignment(srcs, dsts)
    again = ctx.icp_alignment(srcs, dsts)
    for i in range(5):
        single = ctx.icp_alignment([srcs[i]], [dsts[i]])[0]
        for r in (batch[i], again[i]):
            assert np.array_equal(r["T"], single["T"]), "batched result must be bit-identical to the single-pair result"
            assert r["fitness"] == single["fitness"]
            assert r["n_linearize"] == single["n_linearize"]
        # sparse 4-6k-point scans: GICP itself may diverge (pair 4 runs all 32 iterations and ends
        # ~1.8 rad off the ground truth) -- the bar is agreement with the oracle, including there.
        o = oracle.gicp_align(srcs[i], dsts[i])
        rot, trans = synth.se3_error(batch[i]["T"], o["T"])
        assert rot < ROT_TOL and trans < TRANS_TOL
        assert batch[i]["converged"] == o["converged"] and batch[i]["n_linearize"] == o["n_linearize"]


def test_gicp_with_guess_and_cloud_reuse(ctx, oracle, synth, pair5k):
    src, dst, Texp = pair5k
    cs, ct = ctx.create_clouds([src, dst])
    guess = synth.se3(yaw=0.01, t=(0.1, 0.05, 0.0))
    g = ctx.gicp_align([cs], [ct], guesses=[guess])[0]
    o = oracle.gicp_align(src, dst, guess=guess)
    rot, trans = synth.se3_error(g["T"], o["T"])
    assert rot < ROT_TOL and trans < TRANS_TOL
    # aligned output cloud == oracle's fp32 transform of the source, original order
    out = ctx.transform_cloud(cs, g["Tf"])
    ref = oracle.transform_output(g["Tf"], src)
    assert np.array_equal(out, ref)
    cs.destroy(); ct.destroy()


def test_iteration_cap_and_nonconvergence(ctx, oracle, synth, pair5k):
    import b200reg
    src, dst, _ = pair5k
    prm = b200reg.default_params()
    prm.max_iterations = 1
    g = ctx.icp_alignment([src], [dst], params=prm)[0]
    from oracle.oracle import GicpParams
    op = GicpParams.default()
    op.max_iterations = 1
    o = oracle.gicp_align(src, dst, params=op)
    assert g["converged"] == o["converged"] and g["n_linearize"] == o["n_linearize"] == 1
    rot, trans = synth.se3_error(g["T"], o["T"])
    assert rot < ROT_TOL and trans < TRANS_TOL


def test_full_size_100k_tree_equals_bruteforce(ctx, synth):
    """BASELINE config 2 size, no oracle needed: the LBVH traversal must return exactly what the TMA-tiled brute-force
    kernel returns (every one of the 100k points tested for every query) -- indices and fp32 distances bit for bit."""
    src, dst, _ = synth.make_pair(1003, 100000)
    cl, = ctx.create_clouds([dst])
    rng = np.random.default_rng(0)
    far = (src[:3000, :3] + rng.normal(0, 6.0, (3000, 3))).astype(np.float32)
    for q, k in ((dst[::5], 15), (src, 1), (far, 15), (far * np.float32(4.0), 1)):
        ti, td = ctx.knn(cl, q, k)
        bi, bd = ctx.knn(cl, q, k, brute=True)
        assert np.array_equal(td, bd) and np.array_equal(ti, bi)
    cl.destroy()


def test_full_size_100k_properties(ctx, synth):
    """BASELINE config 2 size: size-independent properties instead of an oracle run."""
    src, dst, Texp = synth.make_pair(1000, 100000)
    cs, ct = ctx.create_clouds([src, dst])
    # (1) every point is its own nearest neighbour at distance 0, lists ascending
    idx, d2 = ctx.knn(ct, dst[:30000], 15)
    assert np.array_equal(idx[:, 0], np.arange(30000)) and (d2[:, 0] == 0).all()
    assert (np.diff(d2, axis=1) >= 0).all()
    # (2) k-NN distances equal a numpy recomputation from the returned indices (fp32, same order of ops)
    nb = dst[idx[:2000, 14], :3]
    diff = dst[:2000, :3] - nb
    ref = (diff[:, 0] * diff[:, 0] + diff[:, 1] * diff[:, 1]) + diff[:, 2] * diff[:, 2]
    assert np.array_equal(ref.astype(np.float32), d2[:2000, 14])
    # (3) registration recovers the ground-truth drift correction and is run-to-run bit-identical
    r1 = ctx.gicp_align([cs], [ct])[0]
    r2 = ctx.gicp_align([cs], [ct])[0]
    assert np.array_equal(r1["T"], r2["T"]) and r1["fitness"] == r2["fitness"]
    rot, trans = synth.se3_error(r1["T"], Texp)
    assert r1["converged"] and rot < 3e-3 and trans < 3e-2
    # (4) fitness equals the mean 1-NN d2 of the transformed source (recomputed through the taps)
    moved = ctx.transform_cloud(cs, r1["Tf"])
    _, dd = ctx.knn(ct, moved, 1)
    assert abs(dd.astype(np.float64).mean() - r1["fitness"]) < 1e-9 * max(r1["fitness"], 1e-6)
    cs.destroy(); ct.destroy()


def test_cuda_knn_equals_reference_golden(ctx):
    """Committed answers of the reference's own kd-tree (tests/golden/make_golden.py)."""
    import os
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "knn_ref_nanoflann.npz"))
    cl, = ctx.create_clouds([g["cloud"]])
    for q, k, ik, dk in ((g["q_self"], 15, "idx15", "d15"), (g["q_shift"], 1, "idx1", "d1"), (g["q_shift"][:100], 20, "idx20", "d20")):
        gi, gd = ctx.knn(cl, q, k)
        _tie_ok(gi, gd, g[ik], g[dk])
    cl.destroy()


def test_cuda_gicp_equals_oracle_golden(ctx, synth):
    import os
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "gicp_oracle_3k.npz"))
    cs, ct = ctx.create_clouds([g["src"], g["dst"]])
    ctx.covariances([cs, ct], 15)
    lin = ctx.linearize(cs, ct, np.eye(4))
    assert np.array_equal(lin["corr"], g["corr"]) and np.array_equal(lin["sqd"], g["sqd"])
    assert np.abs(lin["H"] - g["H"]).max() < 1e-9 * np.abs(g["H"]).max()
    r = ctx.gicp_align([cs], [ct])[0]
    rot, tr = synth.se3_error(r["T"], g["T"])
    assert rot < ROT_TOL and tr < TRANS_TOL
    assert r["n_linearize"] == int(g["n_linearize"]) and r["converged"] == bool(g["converged"])
    assert abs(r["fitness"] - float(g["fitness"])) < 1e-6
    cs.destroy(); ct.destroy()


def test_any_k_correspondences(ctx, oracle, pair5k):
    """setCorrespondenceRandomness(k) for k outside the tuned 15/20 (the NanoGICP default ctor uses 20)."""
    src, dst, _ = pair5k
    for k in (5, 12, 20, 27):
        cl, = ctx.create_clouds([dst])
        ctx.covariances([cl], k)
        g = ctx.get_covariances(cl)
        o = oracle.covariances(dst, k)
        err = np.abs(g - o).reshape(len(dst), -1).max(1)
        assert np.median(err) < 1e-11 and np.quantile(err, 0.995) < 1e-5, (k, np.median(err))
        gi, gd = ctx.knn(cl, src[:500], k)
        oi, od = oracle.knn(dst, src[:500], k)
        assert np.array_equal(gi, oi) and np.array_equal(gd, od)
        cl.destroy()


def test_error_paths_return_codes(ctx):
    """Nothing throws across the ABI; bad input is a negative status + message (include/b200reg.h conventions)."""
    import ctypes as C
    import b200reg
    from b200reg import native
    lib = native.lib()
    prm = b200reg.default_params()
    res = (native.Result * 1)()
    pts = np.zeros((10, 4), np.float32)
    ptr = (C.c_void_p * 1)(pts.ctypes.data)
    n0 = (C.c_size_t * 1)(0)
    n10 = (C.c_size_t * 1)(10)
    out = (C.c_void_p * 1)()
    assert lib.b200reg_clouds_create(ctx.h, 1, ptr, n0, C.c_size_t(16), 0, out) == -1            # empty cloud
    assert lib.b200reg_clouds_create(ctx.h, 1, ptr, n10, C.c_size_t(10), 0, out) == -1           # stride not a multiple of 4
    assert lib.b200reg_clouds_create(None, 1, ptr, n10, C.c_size_t(16), 0, out) == -1            # NULL context
    assert b"stride" in lib.b200reg_last_error() or b"bad" in lib.b200reg_last_error()
    cl, = ctx.create_clouds([np.random.default_rng(0).normal(size=(50, 3)).astype(np.float32)])
    arr = (C.c_void_p * 1)(cl.h)
    assert lib.b200reg_clouds_covariances(ctx.h, 1, arr, 0) == -1                                 # k out of range
    assert lib.b200reg_clouds_covariances(ctx.h, 1, arr, 33) == -1
    cov = np.empty((50, 9))
    assert lib.b200reg_get_covariances(ctx.h, cl.h, cov.ctypes.data_as(C.c_void_p)) == -4        # ESTATE: not computed yet
    qp = b200reg.default_quatro_params()
    qp.estimate_scale = 1
    info = (native.QuatroInfo * 1)()
    assert lib.b200reg_quatro_align(ctx.h, 1, arr, arr, C.byref(qp), info, None) == -1            # unsupported mode, loudly
    qp = b200reg.default_quatro_params()
    qp.max_corres = 10000
    assert lib.b200reg_quatro_align(ctx.h, 1, arr, arr, C.byref(qp), info, None) == -1
    cl.destroy()
    with pytest.raises(b200reg.B200RegError):
        b200reg.Context(99)                                                                       # no such device: ENODEV


def test_knn_degenerate_geometries_tie_rule(ctx, oracle):
    """Regular lattices (masses of exactly equal distances), identical points, collinear points, huge offsets:
    the (d2, lower original index) rule must hold everywhere (SURVEY App. A.3)."""
    rng = np.random.default_rng(42)
    g = np.stack(np.meshgrid(np.arange(18), np.arange(18), np.arange(18), indexing="ij"), -1).reshape(-1, 3).astype(np.float32)
    lattice = g[rng.permutation(len(g))] * np.float32(0.5)
    same = np.tile(np.array([[1.5, -2.0, 0.25]], np.float32), (300, 1))
    line = np.c_[np.linspace(0, 50, 2000), np.zeros(2000), np.zeros(2000)].astype(np.float32)
    far = (rng.normal(0, 3, (3000, 3)) + np.array([25000.0, -18000.0, 900.0])).astype(np.float32)
    plane = np.c_[rng.uniform(-20, 20, (4000, 2)), np.zeros(4000)].astype(np.float32)
    for name, pts in (("lattice", lattice), ("identical", same), ("line", line), ("far", far), ("plane", plane)):
        cl, = ctx.create_clouds([pts])
        q = np.concatenate([pts[:400], pts[:200] + np.float32(0.25)])
        for k in (1, 15):
            gi, gd = ctx.knn(cl, q, k)
            oi, od = oracle.knn(pts, q, k, brute=True)
            kk = min(k, len(pts))
            assert np.array_equal(gd[:, :kk], od[:, :kk]), name
            assert np.array_equal(gi[:, :kk], oi[:, :kk]), name
        # covariances stay finite and symmetric even where the neighbourhood is rank deficient
        ctx.covariances([cl], 15)
        c = ctx.get_covariances(cl)
        assert np.isfinite(c).all(), name
        ev = np.linalg.eigvalsh(c[::37])
        assert np.allclose(ev, [1e-3, 1.0, 1.0], atol=1e-6), name
        cl.destroy()


def test_gicp_lattice_pair_with_ties(ctx, oracle, synth):
    """Registration of a lattice against a shifted copy: correspondence ties everywhere, results must still agree."""
    rng = np.random.default_rng(1)
    g = np.stack(np.meshgrid(np.arange(30), np.arange(30), np.arange(4), indexing="ij"), -1).reshape(-1, 3).astype(np.float32)
    dst = (g * np.float32(0.4) + rng.normal(0, 0.01, g.shape).astype(np.float32)).astype(np.float32)
    T = synth.se3(yaw=0.01, t=(0.05, -0.03, 0.01))
    src = synth.to_map_frame(np.c_[dst, np.zeros(len(dst), np.float32)], np.linalg.inv(T))[:, :3]
    r = ctx.icp_alignment([src], [dst])[0]
    o = oracle.gicp_align(src, dst)
    rot, tr = synth.se3_error(r["T"], o["T"])
    assert rot < ROT_TOL and tr < TRANS_TOL
    assert r["n_linearize"] == o["n_linearize"] and r["converged"] == o["converged"]


def test_lm_corner_cases_match_oracle(ctx, oracle, synth, pair5k):
    """State-machine corners: nothing within the correspondence gate (H = 0, zero step, 'converged' like the reference),
    clouds smaller than k, and a single-point target (ill-posed: flags only)."""
    import b200reg
    from oracle.oracle import GicpParams
    src, dst, _ = pair5k
    prm = b200reg.default_params()
    prm.max_corr_dist = 1e-4
    op = GicpParams.default()
    op.max_corr_dist = 1e-4
    g = ctx.icp_alignment([src], [dst], params=prm)[0]
    o = oracle.gicp_align(src, dst, params=op)
    assert np.allclose(g["T"], np.eye(4)) and np.allclose(o["T"], np.eye(4))
    assert g["converged"] == o["converged"] and g["n_linearize"] == o["n_linearize"] and g["n_error"] == o["n_error"]
    assert abs(g["fitness"] - o["fitness"]) < 1e-6 * o["fitness"]
    # n < k: the k-NN list is short, the mean still divides by k (nano_gicp_impl.hpp:320-321)
    tiny = dst[:7]
    cl, = ctx.create_clouds([tiny])
    ctx.covariances([cl], 15)
    assert np.abs(ctx.get_covariances(cl) - oracle.covariances(tiny, 15)).max() < 1e-9
    cl.destroy()
    # (a single-point target makes the rotation unobservable: the LM answer is then dominated by round-off on both
    # sides, so that case is only required to terminate with matching flags)
    g = ctx.icp_alignment([src[:500]], [dst[:1]])[0]
    o = oracle.gicp_align(src[:500], dst[:1])
    assert np.isfinite(g["T"]).all() and g["converged"] == o["converged"]


def test_all_regularization_methods(ctx, oracle, synth, pair5k):
    """setRegularizationMethod: NONE, MIN_EIG, NORMALIZED_MIN_EIG, PLANE, FROBENIUS (nano_gicp_impl.hpp:323-353)."""
    import b200reg
    from oracle.oracle import GicpParams
    src, dst, Texp = pair5k
    cl, = ctx.create_clouds([dst])
    for method in (0, 1, 2, 3, 4):
        ctx.covariances([cl], 15, method)
        g = ctx.get_covariances(cl)
        o = oracle.covariances_ex(dst, 15, method)
        scale = np.abs(o).reshape(len(o), -1).max(1) + 1e-12
        err = np.abs(g - o).reshape(len(o), -1).max(1) / scale
        assert np.median(err) < 1e-10 and np.quantile(err, 0.995) < 1e-5, (method, np.median(err), np.quantile(err, 0.995))
    cl.destroy()
    # the registration honours the method end to end (MIN_EIG here)
    prm = b200reg.default_params()
    prm.regularization = 1
    g = ctx.icp_alignment([src], [dst], params=prm)[0]
    assert g["converged"]
    p3 = ctx.icp_alignment([src], [dst])[0]
    assert not np.array_equal(g["T"], p3["T"])  # a different weighting gives a (slightly) different optimum
    rot, tr = synth.se3_error(g["T"], Texp)
    assert rot < 2e-2 and tr < 0.3  # still lands on the ground truth


def test_large_batch_beyond_the_shared_slot_cache(ctx, synth):
    """More pairs than the LM schedule caches in shared memory (LM_SMEM_SLOTS = 512): the slot list's tail is read from global
    memory; every pair of the batch must equal its single-pair result bit for bit, finished pairs dropping out at
    different steps."""
    rng = np.random.default_rng(7)
    base = [synth.make_pair(1300 + i, 600 + 40 * i, 700 + 30 * i) for i in range(6)]
    order = rng.integers(0, 6, 530)
    srcs = [base[k][0] for k in order]
    dsts = [base[k][1] for k in order]
    batch = ctx.icp_alignment(srcs, dsts)
    singles = [ctx.icp_alignment([b[0]], [b[1]])[0] for b in base]
    assert len({s["n_linearize"] for s in singles}) > 1  # pairs finish at different steps
    for r, k in zip(batch, order):
        assert np.array_equal(r["T"], singles[k]["T"]) and r["fitness"] == singles[k]["fitness"]
        assert r["n_linearize"] == singles[k]["n_linearize"] and r["converged"] == singles[k]["converged"]
