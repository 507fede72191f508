"""The registration's kNN kernel (knn_blocks_kernel) against exhaustive search, through ll_debug_knn_blocks.

ll_knn only runs the unseeded parity kernel.  Every ICP iteration of ll_register runs knn_blocks_kernel instead: the query is transformed in the
kernel from the pose in the device state, the residual-block cap pre-skips features by ICP iteration, and from the second ICP iteration on each
search starts from the previous iteration's 5 neighbours (seeds), which tightens the pruning bound before the first box is opened.  With
LL_KNN_TMA=1 the leaf buckets are staged into shared memory with cp.async.bulk.  The search claims to be exact whatever the seeds and the
variant, so the bar is bit equality with brute force (ids and fp32 squared distances), on the plain and on the TMA-staged context alike.
"""
import ctypes as C

import numpy as np
import pytest

from loam_livox_b200 import synthetic as S

pytestmark = pytest.mark.gpu

IDENT_Q, IDENT_T = np.array([1.0, 0.0, 0.0, 0.0]), np.zeros(3)
BRUTE_PAIRS = 1e9   # above this many point pairs the pinned k-d tree stands in for brute force


def _mk(nc, ns, qc, qs, seed=0):
    mc, ms = S.make_map(nc, ns, seed=S.SEED + seed)
    pose = S.default_pose()
    fc, fs = S.make_features(qc, qs, pose, seed=S.SEED + seed)
    return mc, ms, fc, fs, pose


@pytest.fixture(scope="module")
def contexts():
    """A context on the plain kernel and one on the TMA-staged kernel (LL_KNN_TMA is read once, at ll_ctx_create)."""
    from loam_livox_b200.registration import Context
    out = {}
    with pytest.MonkeyPatch.context() as mp:
        mp.delenv("LL_KNN_TMA", raising=False)
        out["plain"] = Context(0, max_scan_points=100000, max_features=400000)
        mp.setenv("LL_KNN_TMA", "1")
        out["tma"] = Context(0, max_scan_points=100000, max_features=400000)
    yield out
    for c in out.values():
        c.close()


@pytest.fixture(params=["plain", "tma"])
def kctx(request, contexts):
    return request.param, contexts[request.param]


@pytest.fixture(scope="module")
def c2():
    """BASELINE config C2: the 0.5M + 4.5M-point map (four node levels above the buckets) and bench.py's scans."""
    import bench
    return bench.make_inputs(0, "c2")


def _hook(kctx, m, fc, fs, q, t, icp_iter=0, seeds=None, **state):
    from loam_livox_b200.registration import Point_cloud_registration
    kind, ctx = kctx
    reg = Point_cloud_registration(ctx, **state)
    reg.set_pose(q, t)
    idx, d, typ, a3, v3, tma = reg.debug_knn_blocks(m, fc, fs, icp_iter, seeds)
    assert tma == (1 if kind == "tma" else 0), "the context must run the kernel variant it was created for"
    return idx, d, typ, a3, v3


def _ref_knn(oracle, cloud, q, tree=None):
    if tree is None and cloud.shape[0] * q.shape[0] > BRUTE_PAIRS:
        tree = oracle.KdTree(cloud)
    if tree is not None:
        i, d, _ = tree.knn(q, threads=8)
    else:
        i, d, _ = oracle.knn_brute(cloud, q)
    return i, d


def _reference(oracle, mc, ms, fc, fs, q, t, trees=(None, None)):
    """5-NN of every feature at the pose, corner features in the corner cloud, surface features in the surface cloud (slot order)."""
    ic, dc = _ref_knn(oracle, mc, oracle.transform(fc, q, t), trees[0])
    i_s, ds = _ref_knn(oracle, ms, oracle.transform(fs, q, t), trees[1])
    return np.concatenate([ic, i_s]), np.concatenate([dc, ds])


def _assert_rows(idx, d, ri, rd, rows=None, what=""):
    if rows is None:
        rows = np.ones(idx.shape[0], bool)
    bad = np.nonzero(rows & ~((idx == ri).all(1) & (d.view(np.int32) == rd.view(np.int32)).all(1)))[0]
    assert bad.size == 0, f"{what}: {bad.size} of {int(rows.sum())} rows differ from brute force, first {bad[0]}: {idx[bad[0]]} {d[bad[0]]} vs {ri[bad[0]]} {rd[bad[0]]}"


def _feats_at(world, q, t):
    """Scan-frame features that the pose (q, t) puts (to fp32 rounding) at the world points."""
    R = S.quat_to_mat(q)
    f = np.zeros((world.shape[0], 4), np.float32)
    f[:, :3] = ((world[:, :3].astype(np.float64) - t) @ R).astype(np.float32)
    return f


def _shape_queries(P, rng, n_near=96):
    """Features (identity pose) around the cloud P: jittered cloud points, exact cloud points (d = 0), far outside the box, NaN."""
    fin = P[np.isfinite(P[:, :3]).all(1)]
    base = fin if fin.shape[0] else np.zeros((1, 4), np.float32)
    near = base[rng.integers(0, base.shape[0], n_near)].copy()
    near[:, :3] += rng.normal(0, 0.3, (n_near, 3)).astype(np.float32)
    exact = base[rng.integers(0, base.shape[0], 16)].copy()
    far = base[rng.integers(0, base.shape[0], 8)].copy()
    far[:4, 0] += 1000.0
    far[4:, :3] -= 300.0
    nan = near[:4].copy()
    nan[0, 0] = np.nan; nan[1, 1] = np.nan; nan[2, 2] = np.inf; nan[3, :3] = np.nan
    f = np.concatenate([near, exact, far, nan]).astype(np.float32)
    f[:, 3] = 0.0
    finite = np.isfinite(f[:, :3]).all(1)
    return f, finite


def _check_unseeded(kctx, oracle, P, seed, what):
    """Map = (P, P); half the features search the corner tree, half the surface tree, at the identity pose."""
    from loam_livox_b200.registration import Map
    rng = np.random.default_rng(seed)
    f, finite = _shape_queries(P, rng)
    fc, fs = f[::2].copy(), f[1::2].copy()
    fin = np.concatenate([finite[::2], finite[1::2]])
    m = Map(kctx[1], P, P)
    idx, d, typ, _, _ = _hook(kctx, m, fc, fs, IDENT_Q, IDENT_T)
    ri, rd = _reference(oracle, P, P, fc, fs, IDENT_Q, IDENT_T)
    _assert_rows(idx, d, ri, rd, fin, what)
    # non-finite features are not searched: their rows keep the (absent) seeds and NaN distances, and emit no block
    assert (idx[~fin] == -1).all() and np.isnan(d[~fin]).all() and (typ[~fin] == 0).all()
    nfin = int(np.isfinite(P[:, :3]).all(1).sum())
    if nfin < 5:   # fewer than 5 points: -1 / +inf in the missing places
        assert (idx[fin][:, nfin:] == -1).all() and np.isinf(d[fin][:, nfin:]).all()
    m.release()
    return idx, d, fin


# ---------------------------------------------------------------------------------------------- (a) unseeded, at the tree's boundaries
@pytest.mark.parametrize("n", [1, 4, 5, 31, 32, 33, 1023, 1024, 1025, 32769])
def test_unseeded_map_sizes(kctx, oracle, n):
    """Bucket (32 points) and node (32 buckets) boundaries, and maps of fewer than 5 points."""
    rng = np.random.default_rng(100 + n)
    P = np.zeros((n, 4), np.float32)
    P[:, :3] = rng.uniform(-5, 5, (n, 3)).astype(np.float32)
    idx, d, fin = _check_unseeded(kctx, oracle, P, n, f"n={n}")
    exact = np.zeros(fin.shape[0], bool)   # the 16 exact cloud points of _shape_queries sit at rows 96..111 before the split
    order = np.concatenate([np.arange(0, 124, 2), np.arange(1, 124, 2)])
    exact[np.nonzero((order >= 96) & (order < 112))[0]] = True
    assert (d[exact, 0] == 0).all()


def test_unseeded_degenerate_maps(kctx, oracle):
    rng = np.random.default_rng(7)
    # NaN / inf points scattered through the map (the tree indexes the finite ones; ids still refer to the input order)
    P = np.zeros((3000, 4), np.float32)
    P[:, :3] = rng.uniform(-5, 5, (3000, 3)).astype(np.float32)
    P[rng.choice(3000, 300, replace=False), rng.integers(0, 3, 300)] = np.nan
    P[rng.choice(3000, 20, replace=False), 1] = np.inf
    _check_unseeded(kctx, oracle, P, 1, "scattered NaN")
    # all NaN: nothing to find
    idx, d, fin = _check_unseeded(kctx, oracle, np.full((100, 4), np.nan, np.float32), 2, "all NaN")
    assert (idx[fin] == -1).all() and np.isinf(d[fin]).all()
    # zero extent: every point identical, every box a point
    for n in (100, 1100):
        Z = np.tile(np.array([[1.5, -2.0, 0.25, 0.0]], np.float32), (n, 1))
        idx, d, fin = _check_unseeded(kctx, oracle, Z, 3 + n, f"identical x{n}")
        assert (idx[fin] == np.arange(5)).all()
    # 40 exact duplicates scattered over the index range (and so over many buckets): the 5 smallest indices win the tie
    D = np.zeros((5000, 4), np.float32)
    D[:, :3] = rng.uniform(-5, 5, (5000, 3)).astype(np.float32)
    dup = np.sort(rng.choice(5000, 40, replace=False))
    D[dup, :3] = D[dup[17], :3]
    from loam_livox_b200.registration import Map
    m = Map(kctx[1], D, D)
    f = np.repeat(D[dup[17]][None], 8, 0).copy()
    f[4:, :3] += rng.normal(0, 0.01, (4, 3)).astype(np.float32)
    idx, d, _, _, _ = _hook(kctx, m, f[:4], f[4:], IDENT_Q, IDENT_T)
    ri, rd = _reference(oracle, D, D, f[:4], f[4:], IDENT_Q, IDENT_T)
    _assert_rows(idx, d, ri, rd, what="duplicates")
    assert (idx[:4] == dup[:5]).all() and (d[:4] == 0).all()


def test_unseeded_full_size_map(kctx, oracle, c2):
    """The 4.5M-point surface map of config C2 (and its 0.5M-point corner map), sampled queries at a non-trivial pose."""
    from loam_livox_b200.registration import Map
    mc, ms = c2[0], c2[1]
    rng = np.random.default_rng(11)
    pose = S.default_pose()
    wc = mc[rng.integers(0, mc.shape[0], 512)].copy(); wc[:, :3] += rng.normal(0, 0.02, (512, 3)).astype(np.float32)
    ws = ms[rng.integers(0, ms.shape[0], 192)].copy(); ws[:, :3] += rng.normal(0, 0.02, (192, 3)).astype(np.float32)
    fc, fs = _feats_at(wc, pose.q, pose.t), _feats_at(ws, pose.q, pose.t)
    m = Map(kctx[1], mc, ms)
    idx, d, _, _, _ = _hook(kctx, m, fc, fs, pose.q, pose.t)
    m.release()
    ri, rd = _reference(oracle, mc, ms, fc, fs, pose.q, pose.t)   # 192 x 4.5M pairs: still brute force
    _assert_rows(idx, d, ri, rd, what="C2 map")


# ---------------------------------------------------------------------------------------------- (b) the seeds change nothing
def _far_ids(rng, cloud, qw, pool=64):
    """Per query, 5 finite cloud points far from it (the farthest of a random pool)."""
    fin = np.nonzero(np.isfinite(cloud[:, :3]).all(1))[0]
    cand = fin[rng.choice(fin.shape[0], pool, replace=False)]
    dd = ((qw[:, None, :3].astype(np.float64) - cloud[cand][None, :, :3]) ** 2).sum(-1)
    return cand[np.argsort(-dd, axis=1)[:, :5]].astype(np.int32)


def test_seed_invariance(kctx, oracle):
    from loam_livox_b200.registration import Map
    mc, ms, fc, fs, pose = _mk(5000, 45000, 1000, 9000)
    rng = np.random.default_rng(21)
    mc, ms = mc.copy(), ms.copy()
    mc[rng.choice(mc.shape[0], 40, replace=False), 0] = np.nan   # seeds may point at points the tree does not index: they must be ignored
    ms[rng.choice(ms.shape[0], 300, replace=False), 2] = np.nan
    guess = S.perturb_pose(pose, np.random.default_rng(1))
    nc, M = fc.shape[0], fc.shape[0] + fs.shape[0]
    m = Map(kctx[1], mc, ms)
    ri, rd = _reference(oracle, mc, ms, fc, fs, guess.q, guess.t)
    base = _hook(kctx, m, fc, fs, guess.q, guess.t)
    _assert_rows(base[0], base[1], ri, rd, what="no seeds")

    def rand_ids(shape):
        return np.concatenate([rng.integers(0, mc.shape[0], (nc,) + shape[1:]), rng.integers(0, ms.shape[0], (M - nc,) + shape[1:])]).astype(np.int32)
    other = S.Pose(S.quat_mul(guess.q, S.quat_from_euler(*np.radians([1.7, -1.7, 1.7]))), guess.t + np.array([0.3, 0.0, 0.0]))
    moved, _ = _reference(oracle, mc, ms, fc, fs, other.q, other.t)
    rnd = rand_ids((M, 5))
    rnd[::7, 1] = rnd[::7, 0]; rnd[::11, 4] = rnd[::11, 2]   # repeated ids inside a row
    mixed = ri.copy()
    mixed[rng.random((M, 5)) < 0.4] = -1
    mixed[::3, 2] = rand_ids((M,))[::3]
    mixed[::5] = -1
    qw = np.concatenate([oracle.transform(fc, guess.q, guess.t), oracle.transform(fs, guess.q, guess.t)])
    far = np.concatenate([_far_ids(rng, mc, qw[:nc]), _far_ids(rng, ms, qw[nc:])])
    sets = {"true 5-NN": ri, "5-NN 0.3 m / 3 deg away": moved, "random ids": rnd, "ids and -1": mixed, "far points": far,
            "true 5-NN reversed": ri[:, ::-1].copy()}
    for name, seeds in sets.items():
        seeds = np.ascontiguousarray(seeds, np.int32)
        idx, d, typ, a3, v3 = _hook(kctx, m, fc, fs, guess.q, guess.t, icp_iter=1, seeds=seeds)
        _assert_rows(idx, d, ri, rd, what=name)
        assert np.array_equal(typ, base[2]) and np.array_equal(a3, base[3]) and np.array_equal(v3, base[4]), name
    m.release()


def test_seeds_tie_with_zero_extent_boxes(kctx, oracle):
    """200 copies of one point: every box has zero extent and its lower bound equals the seeded 5th distance exactly.  Seeded with the 5 highest
    indices, the search must still open the buckets at lb == d5 and let the lower indices (same distance) displace the seeds."""
    from loam_livox_b200.registration import Map
    P = np.tile(np.array([[0.75, 1.25, -0.5, 0.0]], np.float32), (200, 1))
    rng = np.random.default_rng(5)
    f = np.zeros((64, 4), np.float32)
    f[:, :3] = P[0, :3] + rng.normal(0, 0.5, (64, 3)).astype(np.float32)
    f[:8, :3] = P[0, :3]
    m = Map(kctx[1], P, P)
    ri, rd = _reference(oracle, P, P, f[:32], f[32:], IDENT_Q, IDENT_T)
    assert (ri == np.arange(5)).all()
    for seeds in (np.tile(np.arange(199, 194, -1, dtype=np.int32), (64, 1)), np.tile(np.array([195, 196, 197, 198, 199], np.int32), (64, 1)),
                  np.tile(np.array([3, 199, -1, 100, 0], np.int32), (64, 1))):
        idx, d, _, _, _ = _hook(kctx, m, f[:32], f[32:], IDENT_Q, IDENT_T, icp_iter=1, seeds=seeds)
        _assert_rows(idx, d, ri, rd, what=f"seeds {seeds[0]}")
    m.release()


# ---------------------------------------------------------------------------------------------- (c) the ICP trajectory, replayed
def _trajectory(trace, q_last, t_last):
    """pose_curr of every ICP iteration: iteration 0 at the initial pose, then q_last * q_incre, q_last * t_incre + t_last from the previous
    iteration's increment (x2 = qx, qy, qz, qw, tx, ty, tz)."""
    poses = [(np.asarray(q_last, np.float64), np.asarray(t_last, np.float64))]
    R = S.quat_to_mat(q_last)
    for tr in trace[:-1]:
        x = np.array(list(tr.x2))
        poses.append((S.quat_mul(q_last, np.array([x[3], x[0], x[1], x[2]])), R @ x[4:7] + t_last))
    return poses


@pytest.mark.parametrize("cfg", [(5000, 45000, 1000, 9000), (20000, 180000, 3000, 27000)])
def test_replayed_icp_trajectory(kctx, oracle, cfg):
    """Each ICP iteration of an oracle registration, replayed through the hook and seeded like ll_register seeds it (the previous call's ids)."""
    from loam_livox_b200.registration import Map
    mc, ms, fc, fs, pose = _mk(*cfg)
    guess = S.perturb_pose(pose, np.random.default_rng(0))
    tc, ts = oracle.KdTree(mc), oracle.KdTree(ms)
    p = oracle.default_params(q_w_last=guess.q, t_w_last=guess.t, q_w_curr=guess.q, t_w_curr=guess.t)
    _, _, trace = oracle.register(mc, tc, ms, ts, fc, fs, p, want_trace=True)
    poses = _trajectory(trace, guess.q, guess.t)
    assert len(poses) >= 2
    m = Map(kctx[1], mc, ms)
    seeds = None
    for it, (q, t) in enumerate(poses):
        idx, d, typ, a3, v3 = _hook(kctx, m, fc, fs, q, t, icp_iter=it, seeds=seeds)
        ri, rd = _reference(oracle, mc, ms, fc, fs, q, t, trees=(tc, ts))
        _assert_rows(idx, d, ri, rd, what=f"ICP iteration {it}")
        po = oracle.default_params(q_w_last=guess.q, t_w_last=guess.t, q_w_curr=q, t_w_curr=t)
        blocks, src, _, _ = oracle.build_blocks(mc, tc, ms, ts, fc, fs, po)
        slot = src[:, 1] + np.where(src[:, 0] == 1, fc.shape[0], 0)
        assert np.array_equal(np.nonzero(typ)[0], slot), it
        assert np.array_equal(typ[slot], blocks[:, 0].astype(np.int32) + 1), it
        assert np.array_equal(a3[slot], blocks[:, 4:7]), it
        assert np.allclose(v3[slot], blocks[:, 7:10], rtol=0, atol=1e-15), it
        seeds = idx
    m.release()


# ---------------------------------------------------------------------------------------------- (d) the cap's pre-skip under seeds
@pytest.mark.parametrize("icp_iter", [0, 1, 5])
def test_cap_preskip_keeps_seeds(kctx, oracle, icp_iter):
    """Cap 200, seed 7: a feature of a class of N > 2 cap features is skipped when float(u) * float(N) > float(2 cap), u = ll_cap_uniform(seed,
    ICP iteration, class, index).  Skipped rows return their seeds untouched (NaN distances); searched rows equal brute force."""
    from loam_livox_b200 import capi
    from loam_livox_b200.registration import Map
    mc, ms, fc, fs, pose = _mk(5000, 45000, 1000, 9000)
    cap, seed = 200, 7
    guess = S.perturb_pose(pose, np.random.default_rng(7))
    nc, M = fc.shape[0], fc.shape[0] + fs.shape[0]
    L = capi.lib()
    keep = np.ones(M, bool)
    for cls, (lo, n) in enumerate(((0, nc), (nc, fs.shape[0]))):
        if n > 2 * cap:
            u = np.array([L.ll_cap_uniform(seed, icp_iter, cls, i) for i in range(n)], np.float32)
            keep[lo:lo + n] = ~(u * np.float32(n) > np.float32(2 * cap))
    assert 0 < keep[:nc].sum() < nc and 0 < keep[nc:].sum() < M - nc
    rng = np.random.default_rng(100 + icp_iter)
    seeds = np.concatenate([rng.integers(0, mc.shape[0], (nc, 5)), rng.integers(0, ms.shape[0], (M - nc, 5))]).astype(np.int32)
    seeds[::4, 3:] = -1
    m = Map(kctx[1], mc, ms)
    idx, d, typ, _, _ = _hook(kctx, m, fc, fs, guess.q, guess.t, icp_iter=icp_iter, seeds=seeds, maximum_allow_residual_block=cap, rng_seed=seed)
    m.release()
    active = ~np.isnan(d).all(1)
    assert np.array_equal(active, keep), f"{int((active != keep).sum())} rows disagree with the pre-skip rule"
    assert np.array_equal(idx[~keep], seeds[~keep]) and np.isnan(d[~keep]).all() and (typ[~keep] == 0).all()
    ri, rd = _reference(oracle, mc, ms, fc, fs, guess.q, guess.t)
    _assert_rows(idx, d, ri, rd, keep, f"ICP iteration {icp_iter}")


# ---------------------------------------------------------------------------------------------- (e) motion deblur
def test_deblur_seeded_equals_unseeded(kctx):
    """if_motion_deblur = 1 with a translation increment: the in-kernel interpolated transform moves every query by its own time stamp.  The slots
    and neighbours with seeds equal the unseeded ones bit for bit (the unseeded slots are pinned to the oracle by the deblur block test)."""
    from loam_livox_b200.registration import Map
    mc, ms, fc, fs, pose = _mk(5000, 45000, 1000, 9000)
    rng = np.random.default_rng(9)
    fc, fs = fc.copy(), fs.copy()
    fc[:, 3] = rng.uniform(0.0, 0.1, fc.shape[0]); fs[:, 3] = rng.uniform(0.0, 0.1, fs.shape[0])
    fc[:5, 3] = 0.15; fs[:5, 3] = -0.02
    guess = S.perturb_pose(pose, np.random.default_rng(1))
    kw = dict(if_motion_deblur=1, para_buffer_incremental=[0.0, 0.0, 0.0, 1.0, 0.08, -0.05, 0.02])
    m = Map(kctx[1], mc, ms)
    base = _hook(kctx, m, fc, fs, guess.q, guess.t, **kw)
    assert (base[2] != 0).sum() > 0.5 * base[2].shape[0]
    nc, M = fc.shape[0], fc.shape[0] + fs.shape[0]
    rnd = np.concatenate([rng.integers(0, mc.shape[0], (nc, 5)), rng.integers(0, ms.shape[0], (M - nc, 5))]).astype(np.int32)
    plain = _hook(kctx, m, fc, fs, guess.q, guess.t)[0]   # neighbours without the deblur transform: close, but not the same queries
    for seeds in (base[0], rnd, plain):
        got = _hook(kctx, m, fc, fs, guess.q, guess.t, icp_iter=1, seeds=seeds, **kw)
        for a, b in zip(got, base):
            assert np.array_equal(a, b)
    m.release()


# ---------------------------------------------------------------------------------------------- (f) the TMA-staged kernel end to end
def _reg_tuple(r):
    return (tuple(r.q_w_curr), tuple(r.t_w_curr), r.final_cost, r.icp_iterations, r.corner_used, r.surf_used, r.num_residual_blocks)


@pytest.mark.parametrize("cfg", [(5000, 45000, 1000, 9000), (20000, 180000, 3000, 27000)])
def test_tma_registration_equals_plain(contexts, oracle, cfg):
    """The staged kernel visits the same buckets in the same order, so whole registrations must agree bit for bit with the plain kernel's."""
    from loam_livox_b200.registration import Map, Point_cloud_registration
    mc, ms, fc, fs, pose = _mk(*cfg)
    maps = {k: Map(c, mc, ms) for k, c in contexts.items()}
    tc, ts = oracle.KdTree(mc), oracle.KdTree(ms)
    for seed in range(3):
        guess = S.perturb_pose(pose, np.random.default_rng(seed))
        out = {}
        for k, c in contexts.items():
            reg = Point_cloud_registration(c)
            reg.set_pose(guess.q, guess.t)
            assert reg.find_out_incremental_transfrom(maps[k], fc, fs) == 1
            out[k] = _reg_tuple(reg.result)
        assert out["tma"] == out["plain"], seed
        p = oracle.default_params(q_w_last=guess.q, t_w_last=guess.t, q_w_curr=guess.q, t_w_curr=guess.t)
        ost, ores = oracle.register(mc, tc, ms, ts, fc, fs, p)
        q, t = np.array(out["tma"][0]), np.array(out["tma"][1])
        assert ost == 1 and out["tma"][3] == ores.icp_iterations and out["tma"][4:] == (ores.corner_used, ores.surf_used, ores.num_residual_blocks)
        assert np.linalg.norm(t - np.array(ores.t_w_curr)) < 1e-7 and S.quat_angle(q, np.array(ores.q_w_curr)) < 1e-7
        assert abs(out["tma"][2] - ores.final_cost) <= 1e-7 * ores.final_cost
    for mm in maps.values():
        mm.release()


def test_tma_scan_to_pose_c2_equals_plain(contexts, oracle, c2):
    """bench.py's workload (config C2, scan 0) through ll_scan_to_pose on both kernels: identical results, and within 1e-7 of the oracle."""
    import bench
    from loam_livox_b200 import capi
    from loam_livox_b200.registration import Map, scan_to_pose
    mc, ms, scans, guesses, _ = c2
    pc = capi.PipelineCfg(**bench.PIPE)
    out = {}
    for k, c in contexts.items():
        m = Map(c, mc, ms)
        st = capi.default_reg_state(q_w_last=guesses[0].q, t_w_last=guesses[0].t, q_w_curr=guesses[0].q, t_w_curr=guesses[0].t)
        res, nc, ns = scan_to_pose(c, m, scans[0], 100.0, pc, st)
        m.release()
        assert res.status == 1 and res.registered == 1
        out[k] = _reg_tuple(res) + (nc, ns)
    assert out["tma"] == out["plain"]
    ost, ores, onc, ons = bench.oracle_step(oracle, oracle.Extractor(), (oracle.KdTree(mc), oracle.KdTree(ms)), mc, ms, scans[0], guesses[0], 8)
    r = out["tma"]
    assert ost == 1 and (r[7], r[8]) == (onc, ons) and r[3] == ores.icp_iterations
    assert r[4:7] == (ores.corner_used, ores.surf_used, ores.num_residual_blocks)
    assert np.linalg.norm(np.array(r[1]) - np.array(ores.t_w_curr)) < 1e-7 and S.quat_angle(np.array(r[0]), np.array(ores.q_w_curr)) < 1e-7
    assert abs(r[2] - ores.final_cost) <= 1e-7 * ores.final_cost


# ---------------------------------------------------------------------------------------------- (g) maps and clouds in device memory
def test_device_resident_inputs(kctx, oracle):
    """A map built from CUDA tensors (the streaming mapper's in-place path for XYZI16, the on-device repack for the other two formats) answers like
    the host-built map; ll_transform_dev and ll_voxel_downsample_dev equal the oracle bit for bit."""
    import torch
    from loam_livox_b200 import capi
    from loam_livox_b200.registration import Map
    kind, ctx = kctx
    L = ctx._lib
    mc, ms, fc, fs, pose = _mk(5000, 45000, 1000, 9000)
    guess = S.perturb_pose(pose, np.random.default_rng(2))
    host = Map(ctx, mc, ms)
    want = _hook(kctx, host, fc, fs, guess.q, guess.t)
    rng = np.random.default_rng(3)
    seeds = np.concatenate([rng.integers(0, mc.shape[0], (fc.shape[0], 5)), rng.integers(0, ms.shape[0], (fs.shape[0], 5))]).astype(np.int32)
    want_seeded = _hook(kctx, host, fc, fs, guess.q, guess.t, icp_iter=1, seeds=seeds)
    host.release()

    def pcl32(a):
        o = np.zeros((a.shape[0], 8), np.float32); o[:, :3] = a[:, :3]; o[:, 3] = 1.0; o[:, 4] = a[:, 3]; return o

    def strided(a):   # 18-byte records: x, y, z, intensity float32, then two bytes (a livox_ros_driver PointCloud2 record)
        rec = np.zeros((a.shape[0], 18), np.uint8)
        rec[:, :16] = np.ascontiguousarray(a[:, :4]).view(np.uint8).reshape(-1, 16)
        rec[:, 16] = 7
        return rec
    ctx.set_point_layout(18, 0, 4, 8, 12, capi.LL_I_FLOAT32)
    for fmt, conv in ((capi.LL_FMT_XYZI16, lambda a: np.ascontiguousarray(a)), (capi.LL_FMT_PCL32, pcl32), (capi.LL_FMT_STRIDED, strided)):
        dc, ds = torch.from_numpy(conv(mc)).cuda(), torch.from_numpy(conv(ms)).cuda()
        torch.cuda.synchronize()   # the library's stream does not order against torch's
        h = C.c_void_p()
        ctx.check(L.ll_map_build(ctx.h, C.c_void_p(dc.data_ptr()), mc.shape[0], C.c_void_p(ds.data_ptr()), ms.shape[0], fmt, capi.LL_DEVICE, C.byref(h)))
        m = Map.__new__(Map)
        m.ctx, m.h = ctx, h
        assert (m.size(0), m.size(1)) == (mc.shape[0], ms.shape[0])
        got = _hook(kctx, m, fc, fs, guess.q, guess.t)
        got_seeded = _hook(kctx, m, fc, fs, guess.q, guess.t, icp_iter=1, seeds=seeds)
        ctx.sync()
        del dc, ds
        for a, b in zip(got + got_seeded, want + want_seeded):
            assert np.array_equal(a, b), fmt
        m.release()
    # the documented device-to-device forms
    pts = np.concatenate([fs, fc]).astype(np.float32)
    pts[7, 1] = np.nan
    din = torch.from_numpy(pts).cuda()
    dout = torch.empty_like(din)
    torch.cuda.synchronize()
    q, t = np.ascontiguousarray(guess.q, np.float64), np.ascontiguousarray(guess.t, np.float64)
    ctx.check(L.ll_transform_dev(ctx.h, q.ctypes.data, t.ctypes.data, C.c_void_p(din.data_ptr()), pts.shape[0], C.c_void_p(dout.data_ptr())))
    assert np.array_equal(dout.cpu().numpy(), oracle.transform(pts, guess.q, guess.t), equal_nan=True)
    for leaf in (0.05, 0.4):
        n = C.c_size_t(0)
        dvox = torch.full_like(din, float("nan"))
        torch.cuda.synchronize()
        ctx.check(L.ll_voxel_downsample_dev(ctx.h, C.c_void_p(din.data_ptr()), pts.shape[0], leaf, C.c_void_p(dvox.data_ptr()), C.byref(n)))
        ref = oracle.voxel_grid(pts, leaf)
        assert n.value == ref.shape[0] and np.array_equal(dvox[: n.value].cpu().numpy(), ref), leaf
