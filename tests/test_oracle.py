"""CPU tests of the oracle (oracle/ = restatement of the reference's hot path; test infrastructure, never shipped).

The reference has no tests, fixtures or golden vectors (SURVEY.md §4) and its PCL / Ceres / Eigen dependencies are absent here, so
the oracle is PARITY-UNPINNED with respect to the reference binary.  What pins it instead: independent implementations available
in this image (scipy cKDTree, a NumPy VoxelGrid, central differences, scipy.optimize.least_squares with a per-block Huber) and
the committed golden file (regression pin shared with the GPU tests).
"""
import os
import sys

import numpy as np
import pytest
from scipy.optimize import least_squares
from scipy.spatial import cKDTree

from loam_livox_b200 import synthetic as S

GOLD = os.path.join(os.path.dirname(__file__), "golden", "golden_small.npz")
GOLD_FLANN = os.path.join(os.path.dirname(__file__), "golden", "golden_flann.npz")


# ---------------------------------------------------------------------------------------------- kNN
@pytest.mark.parametrize("n,nq", [(7, 20), (500, 300), (60000, 3000)])
def test_kdtree_matches_brute_force_and_scipy(oracle, n, nq):
    rng = np.random.default_rng(n)
    pts = rng.normal(0, 3, (n, 4)).astype(np.float32)
    q = rng.normal(0, 3, (nq, 4)).astype(np.float32)
    tree = oracle.KdTree(pts)
    idx, d2, found = tree.knn(q)
    bi, bd, bf = oracle.knn_brute(pts, q[:200])
    assert np.array_equal(idx[:200], bi) and np.array_equal(d2[:200], bd) and np.array_equal(found[:200], bf)
    if n >= 5:
        dd, ii = cKDTree(pts[:, :3].astype(np.float64)).query(q[:, :3].astype(np.float64), k=5)
        assert (ii == idx).mean() > 0.999                       # ties aside
        assert np.allclose(dd ** 2, d2, rtol=1e-5, atol=1e-9)   # fp32 accumulation vs fp64


def test_kdtree_ties_and_nonfinite(oracle):
    pts = np.zeros((20, 4), np.float32)
    pts[:10, :3] = 1.0           # 10 identical points: ties resolved by index
    pts[10:15, :3] = np.nan      # skipped, like PCL's convertCloudToArray
    pts[15:, 0] = np.arange(5) + 5.0
    idx, d2, found = oracle.KdTree(pts).knn(np.ones((1, 4), np.float32))
    assert list(idx[0]) == [0, 1, 2, 3, 4] and found[0] == 5 and (d2[0] == 0).all()


# ---------------------------------------------------------------------------------------------- VoxelGrid
def _voxel_numpy(p, leaf):
    """Independent restatement: np.unique on the linearised voxel index, float32 sums in input order."""
    p = p[np.isfinite(p[:, :3]).all(1)]
    inv = np.float32(1.0) / np.float32(leaf)
    mn, mx = p[:, :3].min(0), p[:, :3].max(0)
    min_b = np.floor(mn * inv).astype(np.int64)
    div = np.floor(mx * inv).astype(np.int64) - min_b + 1
    ijk = (np.floor(p[:, :3] * inv) - min_b.astype(np.float32)).astype(np.int64)
    key = ijk[:, 0] + ijk[:, 1] * div[0] + ijk[:, 2] * div[0] * div[1]
    out = []
    for k in np.unique(key):
        sel = p[key == k]
        acc = np.zeros(4, np.float32)
        for row in sel:
            acc = (acc + row).astype(np.float32)
        out.append(acc / np.float32(sel.shape[0]))
    return np.array(out, np.float32)


@pytest.mark.parametrize("n,leaf", [(1, 0.5), (300, 0.4), (3000, 0.2)])
def test_voxel_grid_matches_numpy(oracle, n, leaf):
    rng = np.random.default_rng(n)
    p = rng.uniform(-3, 3, (n, 4)).astype(np.float32)
    if n > 10:
        p[5, 1] = np.nan
    assert np.array_equal(oracle.voxel_grid(p, leaf), _voxel_numpy(p, leaf))


def test_voxel_grid_invariants(oracle):
    rng = np.random.default_rng(2)
    p = rng.uniform(-5, 5, (5000, 4)).astype(np.float32)
    out = oracle.voxel_grid(p, 0.7)
    assert out.shape[0] <= p.shape[0]
    # idempotent up to voxel membership: every output point lies in a distinct voxel
    keys = np.floor(out[:, :3] / np.float32(0.7)).astype(np.int64)
    assert np.unique(keys, axis=0).shape[0] == out.shape[0]
    # centroid of everything is preserved by the weighted mean
    pp = np.abs(p) + 1.0   # one voxel of a 100 m grid
    one = oracle.voxel_grid(pp, 100.0)
    assert one.shape[0] == 1 and np.allclose(one[0], pp.mean(0), atol=1e-3)
    assert oracle.voxel_grid(np.zeros((0, 4), np.float32), 0.5).shape == (0, 4)


# ---------------------------------------------------------------------------------------------- residual models / solver
def _blocks(oracle, nc=150, ns=1350, seed=0):
    mc, ms = S.make_map(2000, 18000, seed=S.SEED + seed)
    pose = S.default_pose()
    fc, fs = S.make_features(nc, ns, pose, seed=S.SEED + seed)
    guess = S.perturb_pose(pose, np.random.default_rng(seed))
    p = oracle.default_params(q_w_last=guess.q, t_w_last=guess.t, q_w_curr=guess.q, t_w_curr=guess.t)
    b, src, ca, sa = oracle.build_blocks(mc, oracle.KdTree(mc), ms, oracle.KdTree(ms), fc, fs, p)
    return b, guess, pose, (mc, ms, fc, fs, p)


def test_jet_jacobian_matches_central_differences(oracle):
    b, guess, _, _ = _blocks(oracle)
    x = oracle.plus([0, 0, 0, 1, 0, 0, 0], [0.01, -0.02, 0.015, 0.05, -0.04, 0.03])
    cost, g, H, r, J = oracle.evaluate(b, guess.q, guess.t, x, want_full=True)
    eps = 1e-6
    for c in range(6):
        d = np.zeros(6)
        d[c] = eps
        rp = oracle.evaluate(b, guess.q, guess.t, oracle.plus(x, d, bound=10.0), want_full=True)[3]
        rm = oracle.evaluate(b, guess.q, guess.t, oracle.plus(x, -d, bound=10.0), want_full=True)[3]
        # residuals are loss-corrected (sqrt(rho') r); compare only blocks in the quadratic zone of the Huber loss
        quad = np.repeat((r.reshape(-1, 3) ** 2).sum(1) < 0.009, 3)
        assert np.allclose(((rp - rm) / (2 * eps))[quad], J[quad, c], atol=2e-6)
    assert np.allclose(H, J.T @ J, rtol=1e-12) and np.allclose(g, J.T @ r, rtol=1e-12)


def test_solver_converges_to_scipy_solution(oracle):
    """Same minimum as an independent trust-region solver on the same objective (Huber applied per 3-vector block)."""
    b, guess, _, _ = _blocks(oracle, seed=3)
    x0 = np.array([0, 0, 0, 1, 0, 0, 0], float)
    xo, so = oracle.solve(b, guess.q, guess.t, x0, 200, bound=10.0)

    a = 0.1

    def fun(d):
        # one scalar per block: sqrt(rho(|r|^2)), so that sum(f^2) = sum(rho) = 2 cost.  |r|^2 is recovered from the loss-corrected
        # residuals the oracle returns (sqrt(rho') r): s~ = rho' s, i.e. s = s~ in the quadratic zone, (s~/a)^2 beyond it.
        rt = oracle.evaluate(b, guess.q, guess.t, oracle.plus(x0, d, bound=10.0), want_full=True)[3].reshape(-1, 3)
        st = (rt ** 2).sum(1)
        sq = np.where(st <= a * a, st, (st / a) ** 2)
        rho = np.where(sq <= a * a, sq, 2 * a * np.sqrt(sq) - a * a)
        return np.sqrt(rho)

    sol = least_squares(fun, np.zeros(6), method="trf", xtol=1e-15, ftol=1e-15, gtol=1e-15, diff_step=1e-7)
    xs = oracle.plus(x0, sol.x, bound=10.0)
    assert abs(0.5 * (sol.fun ** 2).sum() - so["final_cost"]) < 1e-6 * so["final_cost"]
    assert np.allclose(xs, xo, atol=5e-4)   # ceres stops at function_tolerance 1e-6 (relative cost change): flat directions stay loose
    assert so["final_cost"] < so["initial_cost"]


def test_solver_respects_bounds_and_iteration_cap(oracle):
    b, guess, _, _ = _blocks(oracle, seed=4)
    x, s = oracle.solve(b, guess.q, guess.t, [0, 0, 0, 1, 0, 0, 0], 2)
    assert int(s["iterations"]) <= 2
    x, s = oracle.solve(b, guess.q, guess.t, [0, 0, 0, 1, 0, 0, 0], 50, bound=0.01)
    assert np.all(np.abs(x[4:]) <= 0.01 + 1e-15)
    assert abs(np.linalg.norm(x[:4]) - 1.0) < 1e-12


def test_inlier_threshold_is_order_statistic_of_unique_values(oracle):
    r = np.zeros(30)
    r[0::3] = [5, 1, 1, 3, 2, 2, 4, 1, 9, 7]      # L1 norms, with duplicates
    uniq = np.unique(np.abs(r.reshape(-1, 3)).sum(1))
    assert oracle.inlier_threshold(r, 0.8) == uniq[int(0.8 * len(uniq))]


def test_registration_recovers_injected_motion(oracle):
    mc, ms = S.make_map(5000, 45000)
    pose = S.default_pose()
    fc, fs = S.make_features(500, 4500, pose)
    tc, ts = oracle.KdTree(mc), oracle.KdTree(ms)
    for seed in range(3):
        guess = S.perturb_pose(pose, np.random.default_rng(seed))
        p = oracle.default_params(q_w_last=guess.q, t_w_last=guess.t, q_w_curr=guess.q, t_w_curr=guess.t)
        st, res, tr = oracle.register(mc, tc, ms, ts, fc, fs, p, want_trace=True)
        assert st == 1 and res.registered == 1 and 1 <= res.icp_iterations <= 15
        assert np.linalg.norm(np.array(res.t_w_curr) - pose.t) < 5e-3 and S.quat_angle(np.array(res.q_w_curr), pose.q) < 1e-3
        assert all(t.cost2_final <= t.cost2_initial for t in tr)
    # first frames / tiny maps: returns 1 untouched (:199)
    p = oracle.default_params(q_w_last=guess.q, t_w_last=guess.t, q_w_curr=guess.q, t_w_curr=guess.t, current_frame_index=3)
    st, res = oracle.register(mc, tc, ms, ts, fc, fs, p)
    assert st == 1 and res.registered == 0 and np.allclose(res.t_w_curr, guess.t)


# ---------------------------------------------------------------------------------------------- extractor
def test_extractor_masks_and_quirks(oracle):
    raw = S.make_scan(4000, seed=3, zero_frac=0.0, nan_frac=0.0)
    raw[100, :3] = 0.0
    raw[200, :3] = np.nan
    raw[300:303, :3] = 0.0
    ex = oracle.Extractor()
    assert ex.extract(raw, 50.0) > 5
    info = ex.point_info()
    t, lab = info["pt_type"], info["pt_label"]
    assert t[100] & 1 and t[200] & 32 and (t[300:303] & 1).all()
    assert lab[99] & 8 and lab[101] & 8            # near_zero at +-1
    assert lab[98] == -1 and lab[102] == -1        # invalid at +-2
    assert lab[199] & 4 and lab[201] & 4 and lab[198] == -1
    # quirk B17: a bad neighbour at +-1 leaves curvature = |-4 p|^2
    p = raw[99, :3]
    assert np.isclose(info["curvature"][99], np.float32(((np.float32(-4) * p) ** 2).sum()), rtol=1e-6)
    # timestamps: first frame is stamp - (-1) (the reference's uninitialised-first-time quirk), 1e-5 s per point
    assert np.isclose(info["time_stamp"][0], 51.0) and np.isclose(info["time_stamp"][1000] - info["time_stamp"][0], 0.01, atol=1e-4)
    c, s, f = ex.get_features(0.0, 1.0)
    assert c.shape[0] > 0 and s.shape[0] > 1000 and f.shape[0] <= 4000
    assert np.isfinite(c).all() and np.isfinite(s).all()
    # second frame with an older stamp falls back to the last maximum time stamp
    ex.extract(raw, 10.0)
    assert np.isclose(ex.point_info()["time_stamp"][0], np.float32(51.0 + 3999e-5), atol=1e-4)


def test_extractor_too_few_petals_returns_zero(oracle):
    raw = np.zeros((100, 4), np.float32)
    raw[:, 0] = 5.0
    raw[:, 3] = 50.0
    assert oracle.Extractor().extract(raw, 1.0) == 0


# ---------------------------------------------------------------------------------------------- golden regression pin
def test_oracle_reproduces_golden_file(oracle):
    g = np.load(GOLD)
    ex = oracle.Extractor()
    assert ex.extract(g["raw"], 100.0) == int(g["n_scans"])
    info = ex.point_info()
    for k in ("pt_type", "pt_label", "curvature", "view_angle"):
        assert np.array_equal(info[k], g[k], equal_nan=True), k
    c, s, f = ex.get_features(0.0, 1.0)
    assert np.array_equal(c, g["corners"]) and np.array_equal(s, g["surface"])
    assert np.array_equal(oracle.voxel_grid(g["map_surf"], 0.4), g["voxel"])
    ki, kd, _ = oracle.KdTree(g["map_surf"]).knn(g["knn_q"])
    assert np.array_equal(ki, g["knn_idx"]) and np.array_equal(kd, g["knn_d2"])
    p = oracle.default_params(q_w_last=g["guess_q"], t_w_last=g["guess_t"], q_w_curr=g["guess_q"], t_w_curr=g["guess_t"])
    st, res = oracle.register(g["map_corner"], oracle.KdTree(g["map_corner"]), g["map_surf"], oracle.KdTree(g["map_surf"]), g["feat_corner"], g["feat_surf"], p)
    assert st == int(g["reg_status"]) and res.icp_iterations == int(g["reg_iters"])
    assert np.allclose(res.t_w_curr, g["reg_t"], atol=1e-12) and np.allclose(res.q_w_curr, g["reg_q"], atol=1e-12)


# ---------------------------------------------------------------------------------------------- N1: motion deblur (*_mb functors)
def test_mb_jet_jacobian_matches_central_differences(oracle):
    mc, ms = S.make_map(2000, 18000)
    pose = S.default_pose()
    fc, fs = S.make_features(150, 1350, pose)
    fc[:5, 3] = 0.15; fs[:5, 3] = -0.02                                       # s > 1 -> 1.0 ; s < 0 stays negative (refine_blur, :128-141)
    guess = S.perturb_pose(pose, np.random.default_rng(0))
    p = oracle.default_params(q_w_last=guess.q, t_w_last=guess.t, q_w_curr=guess.q, t_w_curr=guess.t, if_motion_deblur=1)
    b, src, ca, sa = oracle.build_blocks(mc, oracle.KdTree(mc), ms, oracle.KdTree(ms), fc, fs, p)
    s = b[:, 10]
    assert s.min() < 0 and s.max() == 1.0 and np.all(s >= -0.3)
    for x in (oracle.plus([0, 0, 0, 1, 0, 0, 0], [0.01, -0.02, 0.015, 0.05, -0.04, 0.03]), np.array([0, 0, 0, 1.0, 0.01, 0.0, -0.02])):   # sin branch, lerp branch
        cost, g, H, r, J = oracle.evaluate(b, guess.q, guess.t, x, want_full=True)
        eps = 1e-6
        quad = np.repeat((r.reshape(-1, 3) ** 2).sum(1) < 0.009, 3)
        for c in range(3, 6):                                                 # translation columns: the slerp branch does not matter
            d = np.zeros(6); d[c] = eps
            rp = oracle.evaluate(b, guess.q, guess.t, oracle.plus(x, d, bound=10.0), want_full=True)[3]
            rm = oracle.evaluate(b, guess.q, guess.t, oracle.plus(x, -d, bound=10.0), want_full=True)[3]
            assert np.allclose(((rp - rm) / (2 * eps))[quad], J[quad, c], atol=2e-6)
        if x[3] < 1.0:                                                        # rotation columns away from the lerp/slerp branch switch
            for c in range(3):
                d = np.zeros(6); d[c] = eps
                rp = oracle.evaluate(b, guess.q, guess.t, oracle.plus(x, d, bound=10.0), want_full=True)[3]
                rm = oracle.evaluate(b, guess.q, guess.t, oracle.plus(x, -d, bound=10.0), want_full=True)[3]
                assert np.allclose(((rp - rm) / (2 * eps))[quad], J[quad, c], atol=5e-6)
        assert np.allclose(H, J.T @ J, rtol=1e-12) and np.allclose(g, J.T @ r, rtol=1e-12)


def test_deblur_registration_recovers_motion_of_distorted_scan(oracle):
    """A scan distorted by the sensor's own motion: with if_motion_deblur = 1 the pose is recovered clearly better than without."""
    mc, ms = S.make_map(5000, 45000)
    tc, ts = oracle.KdTree(mc), oracle.KdTree(ms)
    last = S.default_pose()
    curr = S.Pose(S.quat_mul(last.q, S.quat_from_euler(0.01, -0.02, 0.06)), last.t + np.array([0.20, -0.05, 0.02]))
    fc, fs = S.make_distorted_features(last, curr, 500, 4500)
    errs = {}
    for mode in (0, 1):
        p = oracle.default_params(q_w_last=last.q, t_w_last=last.t, q_w_curr=last.q, t_w_curr=last.t, if_motion_deblur=mode)
        st, res = oracle.register(mc, tc, ms, ts, fc, fs, p)
        assert st == 1 and res.registered == 1
        errs[mode] = (np.linalg.norm(np.array(res.t_w_curr) - curr.t), S.quat_angle(np.array(res.q_w_curr), curr.q))
    assert errs[1][0] < 0.01 and errs[1][1] < 2e-3, errs
    assert errs[1][0] < 0.5 * errs[0][0], errs


# ---------------------------------------------------------------------------------------------- a12 (i): residual-block cap
def test_cap_generator_pinned_between_oracle_and_library(oracle):
    """The counter-based uniform generator that stands in for the reference's std::random_device-seeded m_rand_float (tools_random.hpp:18-25) is
    implemented twice (oracle/orc_registration.hpp, csrc/common.cuh): same bits for every (seed, iteration, stream, index); plausible uniformity."""
    import itertools
    from loam_livox_b200 import capi
    L = capi.lib()   # host-side export, no GPU needed
    for s, it, stream, i in itertools.product((0, 1, -5, 123456789), (0, 1, 7, 14), (0, 1, 2), (0, 1, 2, 999, 30000, 399999)):
        a, b = L.ll_cap_uniform(s, it, stream, i), oracle.lib().orc_cap_uniform(s, it, stream, i)
        assert a == b and 0.0 <= a < 1.0
    u = np.array([L.ll_cap_uniform(3, 0, 2, i) for i in range(20000)])
    assert abs(u.mean() - 0.5) < 0.01 and abs(u.std() - 12 ** -0.5) < 0.01
    assert np.histogram(u, 10, (0, 1))[0].min() > 1800
    # known answers (pins the constants of the hash)
    assert [L.ll_cap_uniform(0, 0, 0, 0), L.ll_cap_uniform(1, 2, 1, 3)] == [0.0, oracle.lib().orc_cap_uniform(1, 2, 1, 3)]


def test_cap_rule_in_the_oracle(oracle):
    """point_cloud_registration.hpp:232-238,339-345,434-458 with the shipped caps (200 / 150): about 2 x cap features of a class survive the pre-skip,
    about cap blocks survive the drop, the registration still converges; a cap above the feature count changes nothing."""
    mc, ms = S.make_map(5000, 45000)
    pose = S.default_pose()
    fc, fs = S.make_features(1000, 9000, pose)
    tc, ts = oracle.KdTree(mc), oracle.KdTree(ms)
    guess = S.perturb_pose(pose, np.random.default_rng(0))
    base = dict(q_w_last=guess.q, t_w_last=guess.t, q_w_curr=guess.q, t_w_curr=guess.t)
    _, full = oracle.register(mc, tc, ms, ts, fc, fs, oracle.default_params(**base))
    _, same = oracle.register(mc, tc, ms, ts, fc, fs, oracle.default_params(maximum_allow_residual_block=10000, rng_seed=9, **base))
    assert np.array_equal(np.array(full.t_w_curr), np.array(same.t_w_curr))
    for cap in (200, 150):
        st, res, tr = oracle.register(mc, tc, ms, ts, fc, fs, oracle.default_params(maximum_allow_residual_block=cap, rng_seed=1, **base), want_trace=True)
        assert st == 1 and 0.7 * 2 * cap < res.surf_used < 1.3 * 2 * cap and 0.7 * 2 * cap < res.corner_used < 1.3 * 2 * cap
        assert all(0.7 * cap < t.blocks_before_select < 1.3 * cap for t in tr)
        assert np.linalg.norm(np.array(res.t_w_curr) - pose.t) < 0.03


# ---------------------------------------------------------------------------------------------- independent witnesses (VERDICT r1, weak #1)
def test_knn_matches_real_flann_kdtree_single_index(oracle):
    """PCL's KdTreeFLANN wraps FLANN's KDTreeSingleIndex (leaf_max_size 15, exact search, sorted).  tests/golden/golden_flann.npz holds the answers of
    the real library (OpenCV's copy of FLANN, cv2.flann algorithm 4, make_golden_flann.py) on a map-like cloud: the oracle's restatement must return the
    same neighbours and the same fp32 squared distances, bit for bit (no exact ties here; FLANN leaves the order of exact ties unspecified, the oracle
    uses the smaller index)."""
    sys.path.insert(0, os.path.join(os.path.dirname(__file__), "golden"))
    import make_golden_flann as G
    g = np.load(GOLD_FLANN)
    (ms, qs), (mc, qc) = G.inputs()
    assert np.array_equal(G.crc([ms, qs, mc, qc]), g["input_crc"]), "the synthetic generator changed: regenerate the fixture"
    for name, cloud, q in (("surf", ms, qs), ("corner", mc, qc)):
        fi, fd = g[f"idx_{name}"], g[f"d2_{name}"]
        oi, od, found = oracle.KdTree(cloud).knn(q)
        assert (found == 5).all()
        assert np.array_equal(fd, od), "fp32 squared distances differ from FLANN's"
        distinct = np.all(np.diff(od, axis=1) > 0, axis=1)
        assert distinct.mean() > 0.99 and np.array_equal(fi[distinct], oi[distinct])
    # the LINEAR index (brute force inside FLANN) as a second witness of the distance arithmetic
    bi, bd, _ = oracle.knn_brute(ms, qc[:200])
    assert np.array_equal(g["linear_d2"], bd)


def test_converged_solution_is_a_stationary_point_of_the_huber_objective(oracle):
    """Independent of the trust-region schedule the restatement follows: restart the solve from its own result until it stops moving; at that point the
    gradient of sum rho(|r_i|^2)/2 in the tangent space (finite differences of the oracle's own cost, NOT its Jacobian code) vanishes to the level the
    function tolerance allows, and no neighbouring point has a lower cost."""
    b, guess, _, _ = _blocks(oracle, seed=5)
    x = np.array([0, 0, 0, 1, 0, 0, 0], float)
    for _ in range(8):
        x, so = oracle.solve(b, guess.q, guess.t, x, 200, bound=10.0)
    cost0 = oracle.evaluate(b, guess.q, guess.t, x)[0]
    h = 1e-6
    g_fd = np.zeros(6)
    for c in range(6):
        e = np.zeros(6); e[c] = h
        g_fd[c] = (oracle.evaluate(b, guess.q, guess.t, oracle.plus(x, e, bound=10.0))[0] - oracle.evaluate(b, guess.q, guess.t, oracle.plus(x, -e, bound=10.0))[0]) / (2 * h)
    _, g, H = oracle.evaluate(b, guess.q, guess.t, x)
    scale = np.sqrt(np.diag(H)) * np.sqrt(2 * cost0)          # |J_c| |f|: the natural size of a gradient component
    assert np.all(np.abs(g_fd) < 1e-4 * scale), (g_fd, scale)
    assert np.allclose(g, g_fd, atol=1e-5 * scale.max())      # and the analytic gradient agrees with the finite differences there
    rng = np.random.default_rng(0)
    for _ in range(50):
        d = rng.normal(0, 1e-4, 6)
        assert oracle.evaluate(b, guess.q, guess.t, oracle.plus(x, d, bound=10.0))[0] >= cost0 * (1 - 1e-9)


# ---------------------------------------------------------------------------------------------- N4: scene alignment (loop-closure reuse of the registration)
def _two_keyframes(seed=0, n_line=4000, n_plane=40000):
    """Line / plane feature clouds of the same scene seen as two keyframes: b = a's scene (another sample) moved by the inverse of (q, t)."""
    al, ap = S.make_map(n_line, n_plane, seed=S.SEED + 50 + seed)
    bl, bp = S.make_map(n_line, n_plane, seed=S.SEED + 60 + seed)
    q = S.quat_from_euler(0.02, -0.015, 0.06)
    t = np.array([0.35, -0.25, 0.1])
    R = S.quat_to_mat(q)
    for c in (bl, bp):
        c[:, :3] = ((c[:, :3].astype(np.float64) - t) @ R).astype(np.float32)    # p_b = R^T (p_a - t)  <=>  p_a = R p_b + t
    return al, ap, bl, bp, q, t


def test_scene_alignment_recovers_the_transform_between_two_keyframes(oracle):
    """Scene_alignment::find_tranfrom_of_two_mappings (scene_alignment.hpp:269-353): three coarse-to-fine registrations with ICP_LINE = 0 on one
    persistent registration object bring keyframe b onto keyframe a."""
    al, ap, bl, bp, q, t = _two_keyframes()
    res, runs = oracle.scene_align(al, ap, bl, bp, threads=4)
    assert runs == 3 and res.registered == 1 and res.status == 1
    assert np.linalg.norm(np.array(res.t_w_curr) - t) < 0.05 and S.quat_angle(np.array(res.q_w_curr), q) < 0.01
    assert res.corner_used == 0 and 3000 < res.num_residual_blocks <= 5000 * 1.3      # ICP_LINE = 0: corners add no residual blocks (:256); the cap of 5000 binds


# ---------------------------------------------------------------------------------------------- committed vectors of round 2
GOLD2 = os.path.join(os.path.dirname(__file__), "golden", "golden_r2.npz")


def test_oracle_reproduces_flann_vectors_and_cap_vectors(oracle):
    """tests/golden/golden_r2.npz: the flann_* arrays were produced by real FLANN (cv2.flann KDTreeSingleIndex, see make_golden_r2.py), the cap_* arrays
    by the oracle; the GPU test of the same name checks the library against the same file."""
    g, s = np.load(GOLD2), np.load(GOLD)
    for name, cloud in (("surf", s["map_surf"]), ("corner", s["map_corner"])):
        oi, od, _ = oracle.KdTree(cloud).knn(s["knn_q"])
        assert np.array_equal(oi, g[f"flann_idx_{name}"]) and np.array_equal(od, g[f"flann_d2_{name}"])
    p = oracle.default_params(q_w_last=g["cap_guess_q"], t_w_last=g["cap_guess_t"], q_w_curr=g["cap_guess_q"], t_w_curr=g["cap_guess_t"],
                              maximum_allow_residual_block=int(g["cap"]), rng_seed=int(g["cap_seed"]))
    tc, ts = oracle.KdTree(g["cap_map_corner"]), oracle.KdTree(g["cap_map_surf"])
    blocks, src, ca, sa = oracle.build_blocks(g["cap_map_corner"], tc, g["cap_map_surf"], ts, g["cap_feat_corner"], g["cap_feat_surf"], p)
    slot = src[:, 1] + np.where(src[:, 0] == 1, g["cap_feat_corner"].shape[0], 0)
    assert np.array_equal(slot, g["cap_slots"]) and (ca, sa) == (int(g["cap_corner_avail"]), int(g["cap_surf_avail"]))
    st, res, tr = oracle.register(g["cap_map_corner"], tc, g["cap_map_surf"], ts, g["cap_feat_corner"], g["cap_feat_surf"], p, want_trace=True)
    assert st == int(g["cap_status"]) and res.icp_iterations == int(g["cap_iters"]) and res.num_residual_blocks == int(g["cap_blocks"])
    assert np.array_equal(np.array([t.blocks_before_select for t in tr]), g["cap_blocks_per_iter"])
    assert np.allclose(res.t_w_curr, g["cap_t"], atol=1e-12) and np.allclose(res.q_w_curr, g["cap_q"], atol=1e-12)
    k = 0
    for sd in (0, 3, -1):
        for it in (0, 5):
            for stream in (0, 1, 2):
                assert [oracle.lib().orc_cap_uniform(sd, it, stream, i) for i in (0, 1, 7, 1000, 399999)] == list(g["cap_uniform"][k])
                k += 1


GOLD_STREAM = os.path.join(os.path.dirname(__file__), "golden", "golden_stream.npz")


@pytest.mark.parametrize("mode,window", [(0, 400), (0, 3), (1, 400)])
def test_oracle_streaming_mapper_reproduces_the_golden_track(oracle, mode, window):
    """tests/golden/golden_stream.npz (make_golden_stream.py): the oracle's process_new_scan loop on a 14-scan sequence -- status, frame index, feature /
    map / append counts and ICP iterations exactly, pose to 1e-9 (OpenMP reduction order) -- in both matching modes and with a window that pops."""
    import zlib
    sys.path.insert(0, os.path.join(os.path.dirname(__file__), "golden"))
    import make_golden_stream as G
    g = np.load(GOLD_STREAM)
    raws = G.scans()
    assert [zlib.crc32(np.ascontiguousarray(r).tobytes()) for r in raws] == [int(x) for x in g["scan_crc"]], "the synthetic generator changed: regenerate the fixture"
    got, want = G.run(mode, window, raws, threads=2), g[f"track_m{mode}_w{window}"]
    assert np.array_equal(got[:, :9], want[:, :9])
    assert np.abs(got[:, 9:] - want[:, 9:]).max() < 1e-9
