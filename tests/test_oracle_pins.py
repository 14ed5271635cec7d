"""Pins of the oracle's association pieces to third-party code.

The reference searches with pcl::KdTreeFLANN<PointXYZI>::nearestKSearch (GLIO/src/Estimator.cpp:3647, :3746, :3832) =
FLANN's KDTreeSingleIndex over L2_Simple<float>, and fits the plane with Eigen's colPivHouseholderQr (:3661).  The kNN
tests compare with FLANN's answers recorded from OpenCV's bundled FLANN (tests/golden/flann_knn5.npz, made by
tests/golden/make_flann_golden.py; the same FLANN code base: KDTREE_SINGLE = KDTreeSingleIndex, LINEAR = brute force; its
L2<float> functor accumulates a 3-vector as ((dx*dx) + dy*dy) + dz*dz, the same order as L2_Simple).  The plane tests
compare with LAPACK's column-pivoted QR (scipy.linalg.qr(pivoting=True) = dgeqp3).  These tests tie the oracle's kNN
(indices AND float distances, bit for bit) and the 5x3 least-squares solve to those libraries."""
import importlib.util
import os

import numpy as np
import pytest

from glio_b200 import synth

HERE = os.path.dirname(os.path.abspath(__file__))


@pytest.fixture(scope="module")
def flann():
    spec = importlib.util.spec_from_file_location("make_flann_golden", os.path.join(HERE, "golden", "make_flann_golden.py"))
    mk = importlib.util.module_from_spec(spec); spec.loader.exec_module(mk)
    return mk, np.load(mk.PATH)


def _assert_is_flanns_answer(flann, name, map_xyz, qry, idx, sqd):
    """idx / sqd equal FLANN's recorded answer for these queries: the sampled rows entry by entry, every row by digest."""
    mk, g = flann
    assert mk.digest(map_xyz, qry) == str(g[name + "_input_sha256"]), f"{name}: not the map / queries FLANN answered"
    rows = g[name + "_rows"]
    assert np.array_equal(idx[rows], g[name + "_idx"]), f"{name}: kNN indices differ from FLANN on the sampled rows"
    assert np.array_equal(sqd[rows], g[name + "_sqd"]), f"{name}: kNN float distances differ from FLANN on the sampled rows"
    assert mk.digest(idx) == str(g[name + "_idx_sha256"]), f"{name}: kNN indices differ from FLANN"
    assert mk.digest(sqd) == str(g[name + "_sqd_sha256"]), f"{name}: kNN float distances differ from FLANN"


def test_knn_matches_flann_kdtree_single_and_linear_small(oracle, flann):
    """Small, dense cloud with many near neighbours: FLANN KDTREE_SINGLE == FLANN LINEAR == oracle brute == oracle kd-tree."""
    map_xyz, pm = flann[0].small_problem()
    ib, db, tie = oracle.knn5_brute(map_xyz, pm)
    assert not tie.any(), "the generator is supposed to be tie free"
    ik, dk = oracle.KdTree(map_xyz).knn5(pm)
    for algo in flann[0].ALGORITHMS:
        _assert_is_flanns_answer(flann, "small_" + algo, map_xyz, pm, ib, db)       # oracle brute force
        _assert_is_flanns_answer(flann, "small_" + algo, map_xyz, pm, ik, dk)       # oracle kd-tree


def test_knn_matches_flann_at_full_map_size(oracle, flann):
    """cfg-2 map (M = 1 M) and 40 k transformed queries of two scans: the oracle's kd-tree (what every full-size parity test
    uses as its reference) returns FLANN KDTreeSingleIndex's indices and float distances bit for bit."""
    map_xyz, qry = flann[0].full_problem()
    tree = oracle.KdTree(map_xyz)
    for k, pm in qry.items():
        ik, dk = tree.knn5(pm)
        _assert_is_flanns_answer(flann, f"full_scan{k}", map_xyz, pm, ik, dk)


def test_assoc_gate_and_indices_consistent_with_flann(oracle, flann):
    """The association's idx5/sqd5 outputs (what the GPU is compared with) are FLANN's, and the radius gate is applied to
    FLANN's 5th SQUARED distance (quirk Q1, Estimator.cpp:3651)."""
    map_xyz, scan, t2, q2 = flann[0].assoc_problem()
    o = oracle.assoc_scan_to_map(map_xyz, scan, t2, q2)
    _assert_is_flanns_answer(flann, "assoc", map_xyz, o["pm"], o["idx5"], o["sqd5"])
    assert np.array_equal(o["status"] == oracle.GO_FAIL_RADIUS, ~(o["sqd5"][:, 4].astype(np.float64) < 1.5))


def test_plane_solve_matches_lapack_pivoted_qr(oracle):
    """colPivHouseholderQr(A).solve(-1) for 5x3 A (Estimator.cpp:3649-3661) against LAPACK dgeqp3 (scipy.linalg.qr with
    pivoting) and against the SVD-based lstsq: <= 1e-12 relative on well-conditioned neighbourhoods, and the same pivot
    choice (largest remaining column norm first)."""
    sl = pytest.importorskip("scipy.linalg")
    rng = np.random.default_rng(5)
    worst = 0.0
    for trial in range(400):
        n = rng.normal(size=3); n /= np.linalg.norm(n)
        c = rng.uniform(-60, 60, 3)
        c += n * (3.0 + abs(rng.normal())) * np.sign(n @ c if n @ c != 0 else 1.0)     # keep the plane away from the origin
        basis = np.linalg.svd(n[None, :])[2][1:]
        A = c + rng.uniform(-0.4, 0.4, (5, 2)) @ basis + 0.02 * rng.normal(size=(5, 1)) * n
        A = A.astype(np.float32).astype(np.float64)
        x, rank = oracle.plane_solve5(A)
        assert rank == 3
        Q, R, piv = sl.qr(A, mode="economic", pivoting=True)
        y = sl.solve_triangular(R, Q.T @ (-np.ones(5)))
        x_qr = np.empty(3); x_qr[piv] = y
        x_ls = np.linalg.lstsq(A, -np.ones(5), rcond=None)[0]
        cond = np.linalg.cond(A)
        tol = 1e-13 * cond                       # backward-stable solvers agree to O(eps * cond)
        worst = max(worst, np.max(np.abs(x - x_qr)) / np.max(np.abs(x_qr)) / max(cond, 1.0))
        assert np.max(np.abs(x - x_qr)) <= tol * np.max(np.abs(x_qr))
        assert np.max(np.abs(x - x_ls)) <= 10 * tol * np.max(np.abs(x_ls))
        # first pivot = the column of largest norm (Eigen and LAPACK agree on this rule)
        assert piv[0] == int(np.argmax(np.linalg.norm(A, axis=0)))
    assert worst < 1e-13


def test_plane_unit_normal_matches_lapack_on_synthetic_neighbourhoods(oracle):
    """End to end on real neighbourhoods of the synthetic map: the oracle's unit normal / offset (Estimator.cpp:3662-3663)
    equal the ones computed from LAPACK's pivoted QR solution to 1e-12."""
    sl = pytest.importorskip("scipy.linalg")
    P = synth.window_problem(W=2, Q=2000, M=30000, seed=9)
    t2, q2 = synth.lidar_pose_in_world(P["poses_init"][0, :3], P["poses_init"][0, 3:])
    o = oracle.assoc_scan_to_map(P["map_xyz"], P["scans"][0], t2, q2)
    ok = np.nonzero(o["status"] != oracle.GO_FAIL_RADIUS)[0][:500]
    for i in ok:
        A = P["map_xyz"][o["idx5"][i]].astype(np.float64)
        Q, R, piv = sl.qr(A, mode="economic", pivoting=True)
        y = sl.solve_triangular(R, Q.T @ (-np.ones(5)))
        x = np.empty(3); x[piv] = y
        nrm = np.linalg.norm(x)
        n_ref, d_ref = x / nrm, 1.0 / nrm
        scale = 1e-13 * np.linalg.cond(A) + 1e-12
        assert np.max(np.abs(o["plane"][i, :3] - n_ref)) <= scale and abs(o["plane"][i, 3] - d_ref) <= scale * max(1.0, abs(d_ref))


def test_oracle_lm_dense_qr_equals_lm_normal_equations(oracle):
    """Levenberg-Marquardt in the oracle (ceres.tgz::internal/ceres/levenberg_marquardt_strategy.cc:69-160): the literal DENSE_QR
    linear solve of [J; D] (the front end's options, LidarOdometry.cpp:521-530) and the normal-equation Cholesky solve give
    the same iterates to rounding, the radius follows Ceres' rule, and the path differs from the dogleg one."""
    P = synth.window_problem(W=1, Q=3000, M=40000, seed=synth.SEED0 + 9)
    ident_q, zero_t = [1.0, 0.0, 0.0, 0.0], [0.0, 0.0, 0.0]
    t2, q2 = synth.lidar_pose_in_world(P["poses_init"][0, :3], P["poses_init"][0, 3:7])
    state = np.concatenate([t2, q2])[None, :]
    prm = oracle.default_params(); prm.kd_max_radius = 1.0; prm.surf_dist_thres = 0.06; prm.weight_min = 0.4; prm.lidar_const = 1.0
    o = oracle.assoc_scan_to_map(P["map_xyz"], P["scans"][0], t2, q2, prm=prm)
    v = o["status"] == oracle.GO_VALID
    kf = np.zeros(int(v.sum()), np.int32); ones = np.ones(int(v.sum()))
    prob = oracle.WindowProblem(state, None, ident_q, zero_t, huber_delta=0.1)
    prob.add_unary(kf, P["scans"][0][v], o["nsd"][v], ones)
    res = {}
    for strat in (0, 1, 2):
        prob.reset_state(state)
        res[strat] = prob.solve(oracle.solver_options(reserved=strat, max_num_iterations=8), mode=0)
    a, b = res[1], res[2]
    assert a["summary"].num_iterations == b["summary"].num_iterations >= 3
    for x, y in zip(a["steps"], b["steps"]):
        assert np.max(np.abs(x - y)) <= 1e-9
    for ia, ib in zip(a["iterations"], b["iterations"]):
        assert ia["step_is_successful"] == ib["step_is_successful"]
        assert ia["trust_region_radius"] == pytest.approx(ib["trust_region_radius"], rel=1e-8)
    # Ceres' rule on the accepted steps: radius_{k+1} = min(max_radius, radius_k / max(1/3, 1 - (2 rho - 1)^3))
    its = a["iterations"]
    for prev, cur in zip(its, its[1:]):
        if cur["step_is_successful"]:
            want = min(1e16, prev["trust_region_radius"] / max(1.0 / 3.0, 1.0 - (2.0 * cur["relative_decrease"] - 1.0) ** 3))
            assert cur["trust_region_radius"] == pytest.approx(want, rel=1e-12)
    assert a["summary"].final_cost < 0.7 * a["summary"].initial_cost
    # a different algorithm from the dogleg one: the first steps are not the same vector
    assert np.max(np.abs(res[0]["steps"][0] - a["steps"][0])) > 1e-9
