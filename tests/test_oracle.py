"""CPU tests of the oracle (test infrastructure) -- run with -m "not gpu".

The oracle is pinned three ways: (1) its k-NN against the REFERENCE's own kd-tree (golden answers
generated from third_party/nano_gicp/.../nanoflann_impl.hpp through oracle/_ref, tests/golden/make_golden.py);
(2) closed-form known answers for the covariance / SE(3) pieces; (3) ground-truth recovery.
"""
import os

import numpy as np

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def _tie_ok(idx_g, d2_g, idx_o, d2_o):
    assert np.array_equal(d2_g, d2_o)
    rows, cols = np.nonzero(idx_g != idx_o)
    for r, c in zip(rows, cols):
        assert (c > 0 and d2_o[r, c - 1] == d2_o[r, c]) or (c + 1 < d2_o.shape[1] and d2_o[r, c + 1] == d2_o[r, c])


def test_oracle_knn_equals_reference_nanoflann_golden(oracle):
    g = np.load(os.path.join(GOLD, "knn_ref_nanoflann.npz"))
    for q, k, ik, dk in ((g["q_self"], 15, "idx15", "d15"), (g["q_shift"], 1, "idx1", "d1"), (g["q_shift"][:100], 20, "idx20", "d20")):
        idx, d2 = oracle.knn(g["cloud"], q, k)
        _tie_ok(idx, d2, g[ik], g[dk])
        bi, bd = oracle.knn(g["cloud"], q, k, brute=True)
        assert np.array_equal(idx, bi) and np.array_equal(d2, bd)


def test_oracle_knn_equals_live_reference_nanoflann(oracle, synth):
    """The reference kd-tree's answers on seeded samples of these query sets, and the oracle's registration with that
    kd-tree behind its kNN, are stored in golden/knn_ref_nanoflann_6k.npz (make_golden.py ref_samples)."""
    g = np.load(os.path.join(GOLD, "knn_ref_nanoflann_6k.npz"))
    src, dst, _ = synth.make_pair(77, 6000, 7000)
    for name, q, k in (("self15", dst[:2000], 15), ("src1", src, 1), ("shift15", src[:500] + np.float32(2.5), 15)):
        oi, od = oracle.knn(dst, q[g["rows_" + name]], k)
        _tie_ok(oi, od, g["idx_" + name], g["d2_" + name])
    # the switchable backend gives the same registration (H/b sums follow the OpenMP guided schedule
    # like the reference's, nano_gicp_impl.hpp:225,256-266, so only round-off may differ)
    a = oracle.gicp_align(src, dst)
    assert np.abs(a["T"] - g["T_ref_backend"]).max() < 1e-9 and a["fitness"] == float(g["fitness_ref_backend"])


def test_covariance_of_a_plane_is_closed_form(oracle):
    """Points on z = 0.3x - 0.2y + 1: PLANE regularisation gives I - (1 - 1e-3) n n^T (nano_gicp_impl.hpp:341-352)."""
    rng = np.random.default_rng(0)
    xy = rng.uniform(-5, 5, (4000, 2))
    pts = np.c_[xy, 0.3 * xy[:, 0] - 0.2 * xy[:, 1] + 1.0].astype(np.float32)
    n = np.array([0.3, -0.2, -1.0])
    n /= np.linalg.norm(n)
    want = np.eye(3) - (1 - 1e-3) * np.outer(n, n)
    cov = oracle.covariances(pts, 15)
    assert np.abs(cov - want).max() < 2e-5  # fp32 input quantisation of the plane
    ev = np.linalg.eigvalsh(cov[::100])
    assert np.allclose(ev, [1e-3, 1, 1], atol=1e-9)


def test_query_transform_order_and_output_transform(oracle):
    rng = np.random.default_rng(2)
    pts = rng.normal(0, 30, (1000, 3)).astype(np.float32)
    T = np.eye(4)
    a = 0.3
    T[:3, :3] = [[np.cos(a), -np.sin(a), 0], [np.sin(a), np.cos(a), 0], [0, 0, 1]]
    T[:3, 3] = [1.5, -2.25, 0.125]
    Tf = T.astype(np.float32)
    x, y, z = pts[:, 0], pts[:, 1], pts[:, 2]
    seq = np.stack([((Tf[r, 0] * x + Tf[r, 1] * y) + Tf[r, 2] * z) + Tf[r, 3] for r in range(3)], 1)
    right = np.stack([Tf[r, 0] * x + (Tf[r, 1] * y + (Tf[r, 2] * z + Tf[r, 3])) for r in range(3)], 1)
    assert np.array_equal(oracle.transform_queries(T, pts), seq)      # SURVEY App. A.4
    assert np.array_equal(oracle.transform_output(Tf, pts), right)    # PCL SSE order, App. B.2/B.3


def test_gicp_recovers_exact_rigid_motion(oracle, synth):
    """Same physical points seen from a shifted frame: LM must land on the exact transform."""
    _, dst, _ = synth.make_pair(5, 4000, 4000)
    T = synth.se3(yaw=0.03, pitch=0.004, roll=-0.006, t=(0.25, -0.15, 0.04))
    src = synth.to_map_frame(dst, np.linalg.inv(T))
    r = oracle.gicp_align(src, dst)
    rot, tr = synth.se3_error(r["T"], T)
    assert r["converged"] and rot < 2e-5 and tr < 5e-4
    assert r["fitness"] < 1e-6


def test_config1_single_10k_pair_on_cpu(oracle, synth):
    """BASELINE.json configs[0]: one Nano-GICP align of two 10k-point synthetic scans on the CPU path."""
    src, dst, Texp = synth.make_pair(1000, 10000)
    r = oracle.gicp_align(src, dst, want_trace=True)
    rot, tr = synth.se3_error(r["T"], Texp)
    assert r["converged"] and not r["lm_failed"]
    assert rot < 5e-3 and tr < 2e-2
    assert r["n_linearize"] == len(r["trace"]) and r["iterations"] == r["n_linearize"] - 1
    y0 = r["trace"][:, 58]
    assert (np.diff(y0) < 0).all()  # the LM objective decreases at every accepted step


def test_oracle_matches_committed_golden(oracle):
    g = np.load(os.path.join(GOLD, "gicp_oracle_3k.npz"))
    src, dst = g["src"], g["dst"]
    cov_s, cov_t = oracle.covariances(src, 15), oracle.covariances(dst, 15)
    assert np.abs(cov_s[::60] - g["cov_src_sample"]).max() < 1e-12
    assert np.abs(cov_t[::70] - g["cov_tgt_sample"]).max() < 1e-12
    lin = oracle.linearize(src, dst, cov_s, cov_t, np.eye(4))
    assert np.array_equal(lin["corr"], g["corr"]) and np.array_equal(lin["sqd"], g["sqd"])
    assert np.abs(lin["H"] - g["H"]).max() < 1e-9 * np.abs(g["H"]).max()
    r = oracle.gicp_align(src, dst)
    assert np.abs(r["T"] - g["T"]).max() < 1e-9
    assert r["n_linearize"] == int(g["n_linearize"]) and r["converged"] == bool(g["converged"])
    assert abs(r["fitness"] - float(g["fitness"])) < 1e-12


def test_lm_state_machine_edge_cases(oracle, synth):
    from oracle.oracle import GicpParams
    src, dst, _ = synth.make_pair(6, 2000, 2000)
    p = GicpParams.default()
    p.max_iterations = 1
    r = oracle.gicp_align(src, dst, params=p)
    assert r["n_linearize"] == 1 and r["iterations"] == 0
    p = GicpParams.default()
    p.max_corr_dist = 1e-4  # nothing matches: H = 0, the step is zero, delta = I => "converged" like the reference
    r = oracle.gicp_align(src, dst, params=p)
    assert np.allclose(r["T"], np.eye(4))


def test_quatro_matchers_known_answers(oracle, synth):
    """Matcher::optimizedMatching / advancedMatching restatements on a small pair: structural properties the reference's
    code guarantees (matcher.cc:118-356, 358-561), plus the planted motion recovered by the QUATRO solve from either."""
    src, dst, Texp = synth.make_pair(2000, 8000, 9000, mode="quatro")
    _, _, fs = oracle.fpfh(src)
    _, _, fd = oracle.fpfh(dst)
    adv = oracle.match_advanced(src, dst, fs, fd)
    cross = oracle.match_advanced(src, dst, fs, fd, tuple_test=False)
    opt, mutual = oracle.match(src, dst, fs, fd)
    # sorted + unique (src, dst) pairs (matcher.cc:353-355); the tuple test only removes cross-checked pairs
    key = lambda c: c[:, 0].astype(np.int64) * (1 << 32) + c[:, 1]
    assert np.all(np.diff(key(adv)) > 0) and np.all(np.diff(key(cross)) > 0)
    assert set(map(tuple, adv)) <= set(map(tuple, cross))
    # the cross check is a bijection between the matched subsets
    assert len(set(cross[:, 0])) == len(cross) == len(set(cross[:, 1]))
    # swapping the arguments swaps the columns (fi/fj swap, matcher.cc:125-130): same set of physical pairs
    adv_sw = oracle.match_advanced(dst, src, fd, fs)
    assert set(map(tuple, adv_sw[:, ::-1])) == set(map(tuple, adv))
    # optimizedMatching: gated + capped at max_corres + 3 (break AFTER exceeding, matcher.cc:537)
    assert 0 < len(opt) <= 203 and len(mutual) >= len(opt)
    # both correspondence sets put the solver inside the refinement's basin of the planted motion
    for corr in (adv, opt):
        r = oracle.quatro_solve(src, dst, corr)
        rot, tr = synth.se3_error(r["T"], Texp)
        assert r["valid"] and rot < 0.06 and tr < 3.5, (len(corr), rot, tr)


def test_quatro_oracle_matches_committed_golden(oracle):
    """Guards the (reference-unpinned) Quatro restatement against silent drift: tests/golden/quatro_oracle_2k.npz."""
    g = np.load(os.path.join(GOLD, "quatro_oracle_2k.npz"))
    ns, _, fs = oracle.fpfh(g["src"])
    _, _, fd = oracle.fpfh(g["dst"])
    assert np.array_equal(np.isnan(ns[::25]), np.isnan(g["normals_src_sample"]))
    assert np.nanmax(np.abs(ns[::25] - g["normals_src_sample"])) < 1e-6
    assert np.abs(fs[::25] - g["fpfh_src_sample"]).max() < 1e-4 and np.abs(fd[::25] - g["fpfh_dst_sample"]).max() < 1e-4
    opt, mutual = oracle.match(g["src"], g["dst"], fs, fd)
    adv = oracle.match_advanced(g["src"], g["dst"], fs, fd)
    assert np.array_equal(opt, g["corr_opt"]) and len(mutual) == int(g["n_mutual"]) and np.array_equal(adv, g["corr_adv"])
    for corr, T, clique, gnc in ((opt, g["T_opt"], g["clique_opt"], g["gnc_opt"]), (adv, g["T_adv"], g["clique_adv"], g["gnc_adv"])):
        r = oracle.quatro_solve(g["src"], g["dst"], corr)
        assert np.array_equal(r["clique"], clique) and r["gnc_iters"] == int(gnc)
        assert np.abs(r["T"] - T).max() < 1e-9
