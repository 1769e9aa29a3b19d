"""GPU-vs-oracle parity at the BASELINE sizes (SURVEY.md §8(d): N = M = 100 000): LoopClosure::icpAlignment
(nano_gicp_impl.hpp:173-357 behind loop_closure.cpp:110-136) and LoopClosure::coarseToFineAlignment
(loop_closure.cpp:138-159) on raw 100k-point scans and on their 0.3 m voxelised variant, with the oracle's kNN routed
through the reference's own nanoflann (oracle/_ref) when it is built.

Bars (BASELINE.json north_star): correspondence indices bit-exact, SE(3) within 1e-4 rad / 1e-3 m, iteration counters
and flags equal.
"""
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROT_TOL, TRANS_TOL = 1e-4, 1e-3


@pytest.fixture(scope="module")
def ref_oracle(oracle):
    """The oracle with the reference's kd-tree behind its kNN (falls back to the oracle's own tree if _ref is missing)."""
    pinned = os.path.exists(oracle.ref_so_path()) and oracle.use_ref_nanoflann(True) == 0
    yield oracle, pinned
    oracle.use_ref_nanoflann(False)


@pytest.mark.parametrize("seed", [1000, 1001, 1002])
def test_icp_alignment_100k_matches_oracle(ctx, ref_oracle, synth, seed):
    oracle, _ = ref_oracle
    src, dst, Texp = synth.make_pair(seed, 100000, 100000)
    assert len(src) == 100000 and len(dst) == 100000
    g = ctx.icp_alignment([src], [dst])[0]
    o = oracle.gicp_align(src, dst)
    rot, trans = synth.se3_error(g["T"], o["T"])
    assert rot < ROT_TOL and trans < TRANS_TOL, (seed, rot, trans)
    assert g["converged"] == o["converged"] and g["iterations"] == o["iterations"]
    assert g["n_linearize"] == o["n_linearize"] and g["n_error"] == o["n_error"]
    assert abs(g["fitness"] - o["fitness"]) < 1e-5 * max(o["fitness"], 1e-3)
    # RegistrationOutput::pose_between_eig_ (loop_closure.cpp:129-134)
    want = g["Tf"].astype(np.float64) if g["valid"] else np.eye(4)
    assert np.array_equal(g["pose_between"], want)
    # correspondences of the FIRST linearize (identity guess): indices and fp32 distances bit-exact at full size
    cs, ct = ctx.create_clouds([src, dst])
    ctx.covariances([cs, ct], 15)
    lin = ctx.linearize(cs, ct, np.eye(4))
    ol = oracle.linearize(src, dst, ctx.get_covariances(cs), ctx.get_covariances(ct), np.eye(4))
    assert np.array_equal(lin["corr"], ol["corr"]), "correspondence indices must be bit-exact at 100k x 100k"
    assert np.array_equal(lin["sqd"], ol["sqd"])
    assert np.abs(lin["H"] - ol["H"]).max() < 1e-9 * np.abs(ol["H"]).max()
    # ... and at the converged pose (the last linearize of the solve sees this neighbourhood)
    lin = ctx.linearize(cs, ct, g["T"])
    ol = oracle.linearize(src, dst, ctx.get_covariances(cs), ctx.get_covariances(ct), g["T"])
    assert np.array_equal(lin["corr"], ol["corr"]) and np.array_equal(lin["sqd"], ol["sqd"])
    cs.destroy(); ct.destroy()
    rot, trans = synth.se3_error(g["T"], Texp)
    assert rot < 3e-3 and trans < 3e-2, ("ground truth", rot, trans)


def test_covariances_100k_match_oracle(ctx, ref_oracle, synth):
    oracle, _ = ref_oracle
    _, dst, _ = synth.make_pair(1001, 100000, 100000)
    cl, = ctx.create_clouds([dst])
    ctx.covariances([cl], 15)
    g = ctx.get_covariances(cl)
    o, knn = oracle.covariances(dst, 15, return_knn=True)
    err = np.abs(g - o).reshape(len(dst), -1).max(1)
    assert np.median(err) < 1e-12 and np.quantile(err, 0.999) < 1e-6, (np.median(err), np.quantile(err, 0.999))
    gi, gd = ctx.knn(cl, dst[::7], 15)
    assert np.array_equal(gi, knn[::7]), "15-NN index lists must be bit-exact at 100k"
    # the reference kd-tree's own lists on a seeded sample of these queries (tests/golden/make_golden.py ref_samples)
    ref = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "knn_ref_nanoflann_100k.npz"))
    assert np.array_equal(gi[ref["rows_self15"]], ref["idx_self15"]), "15-NN index lists must equal the reference kd-tree's"
    cl.destroy()


def test_compute_error_tap_matches_oracle(ctx, oracle, synth, pair20k):
    """NanoGICP::compute_error in isolation (row a7, nano_gicp_impl.hpp:272-296): stale correspondences and Mahalanobis
    matrices from a linearize at T_lin, the error sum at several trial poses."""
    src, dst, _ = pair20k
    cs, ct = ctx.create_clouds([src, dst])
    ctx.covariances([cs, ct], 15)
    cov_s, cov_t = ctx.get_covariances(cs), ctx.get_covariances(ct)
    T_lin = synth.se3(yaw=0.004, t=(0.05, -0.02, 0.01))
    for T_trial in (T_lin, np.eye(4), synth.se3(yaw=0.02, pitch=-0.004, t=(0.3, -0.2, 0.05)), synth.se3(roll=0.01, t=(-1.0, 0.4, 0.0))):
        g = ctx.compute_error(cs, ct, T_lin, T_trial)
        o = oracle.compute_error(src, dst, cov_s, cov_t, T_lin, T_trial)
        assert abs(g - o) < 1e-9 * abs(o), (g, o)
    # at T_trial == T_lin it is the linearize pass's own error sum
    lin = ctx.linearize(cs, ct, T_lin)
    assert abs(ctx.compute_error(cs, ct, T_lin, T_lin) - lin["err"]) < 1e-12 * abs(lin["err"])
    # a tight gate drops correspondences on both sides alike
    g = ctx.compute_error(cs, ct, np.eye(4), T_lin, max_corr_dist=0.25)
    o = oracle.compute_error(src, dst, cov_s, cov_t, np.eye(4), T_lin, max_corr_dist=0.25)
    assert abs(g - o) < 1e-9 * abs(o)
    cs.destroy(); ct.destroy()


def _check_loop_closure(ctx, oracle, synth, src, dst, Texp, tag):
    res, qi = ctx.loop_closure([src], [dst])
    r, q = res[0], qi[0]
    assert q["valid"], tag
    # (a) the fine stage on the SAME coarse transform: the parity bar
    o_same = oracle.coarse_to_fine(src, dst, quatro_T=q["T"])
    rot, tr = synth.se3_error(r["T"], o_same["T"])
    assert rot < ROT_TOL and tr < TRANS_TOL, (tag, rot, tr)
    assert r["converged"] == o_same["converged"]
    assert r["n_linearize"] == o_same["gicp"]["n_linearize"] and r["n_error"] == o_same["gicp"]["n_error"]
    assert abs(r["fitness"] - o_same["fitness"]) < 1e-5 * max(o_same["fitness"], 1e-3)
    # (b) RegistrationOutput::pose_between_eig_ = fine (float -> double) * quatro (loop_closure.cpp:156)
    if r["valid"]:
        assert np.abs(r["pose_between"] - r["T"]).max() == 0.0
    rot, tr = synth.se3_error(r["T"], Texp)
    assert rot < 5e-3 and tr < 5e-2, (tag, "ground truth", rot, tr)
    return r, q


@pytest.mark.parametrize("seed", [2000, 2001, 2002])
def test_loop_closure_100k_voxelised_matches_oracle(ctx, ref_oracle, synth, seed):
    """configs[2] at the reference-realistic size: 100k raw returns voxelised at 0.3 m (setSrcAndDstCloud, loop_closure.cpp:107)."""
    oracle, _ = ref_oracle
    src, dst, Texp = synth.make_pair(seed, 100000, 100000, mode="quatro", voxel=0.3)
    r, q = _check_loop_closure(ctx, oracle, synth, src, dst, Texp, ("voxel", seed))
    # the two COMPLETE pipelines (each with its own Quatro stage) land within Nano-GICP's stopping tolerance
    o = oracle.coarse_to_fine(src, dst)
    assert o["quatro"]["valid"]
    rot, tr = synth.se3_error(r["T"], o["T"])
    assert rot < 2e-3 and tr < 1e-2, ("pipelines", seed, rot, tr)


def test_loop_closure_100k_raw_matches_oracle(ctx, ref_oracle, synth):
    """configs[2] on RAW 100k x 100k scans (no voxel grid): FPFH over ~1000-neighbour balls, 1e10 descriptor pairs."""
    oracle, _ = ref_oracle
    src, dst, Texp = synth.make_pair(2000, 100000, 100000, mode="quatro")
    assert len(src) == 100000 and len(dst) == 100000
    _check_loop_closure(ctx, oracle, synth, src, dst, Texp, "raw")


def test_invalid_fine_stage_keeps_identity_times_quatro(ctx, synth, native):
    """loop_closure.cpp:129-134,156: when the fine stage is not valid its pose_between_eig_ stays Identity and the
    composed output is I * T_quatro -- not the solver's last pose."""
    src, dst, _ = synth.make_pair(2000, 30000, 30000, mode="quatro", voxel=0.3)
    gp = native.default_params()
    gp.icp_score_thr = 1e-9  # nothing passes the score gate
    res, qi = ctx.loop_closure([src], [dst], gparams=gp)
    r, q = res[0], qi[0]
    assert q["valid"] and r["converged"] and not r["valid"]
    assert np.array_equal(r["pose_between"], q["T"])
    assert not np.array_equal(r["T"], q["T"])  # the telemetry field still carries solver * coarse
    # icpAlignment alone: Identity
    g = ctx.icp_alignment([src], [dst], params=gp)[0]
    assert not g["valid"] and np.array_equal(g["pose_between"], np.eye(4))
