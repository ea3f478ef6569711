"""Pins oracle/icp_oracle.c against the reference's OWN code: oracle/_ref/libicp_ref.so is the
reference's headers (ICP_REFERENCE_ROOT/icp-variants/*.h) compiled where they lie against the
stand-ins of oracle/ref_shim/ (Eigen / FLANN / Ceres / PCL are not installed; see
oracle/ref_driver.cpp for what that does and does not pin).

Bit-exact: transforms, correspondence indices (3-D, 6-D, projective incl. its unsigned wrap),
weights, rejection, pyramid levels, mt19937 selection, the LM path (same trust-region restatement
driving the reference's own functors).  Tolerance 1e-5 rad / 1e-5 m (BASELINE.json north_star):
the linear solvers, where the reference solves the 4M x 6 system in fp32 (SVD / LU) and the
oracle accumulates the 6x6 normal equations in fp64.
"""
import os

import numpy as np
import pytest

from oracle import oracle as O
from oracle import ref as R

pytestmark = pytest.mark.skipif(not R.available(), reason="neither the reference sources (ICP_REFERENCE_ROOT) nor a prebuilt oracle/_ref/libicp_ref.so")

ROT_TOL = 1e-5   # rad
TRANS_TOL = 1e-5  # m
MINF = -np.inf


def rot_err(a, b):
    return 2.0 * np.arcsin(min(1.0, np.linalg.norm(a[:3, :3].astype(np.float64) - b[:3, :3]) / (2.0 * np.sqrt(2.0))))


def _pose(seed=0, t=0.05, deg=4.0):
    from icp_variants_b200.synth import make_pose
    rng = np.random.default_rng(seed)
    return make_pose(rng.uniform(-t, t, 3), rng.uniform(-deg, deg, 3))


def _cloud(n, seed, quant=None, nonfinite=0):
    rng = np.random.default_rng(seed)
    p = rng.uniform(-1, 1, (n, 3)).astype(np.float32)
    if quant:
        p = (np.round(p * quant) / quant).astype(np.float32)   # many exact ties / duplicates
    nrm = rng.normal(size=(n, 3)).astype(np.float32)
    nrm /= np.linalg.norm(nrm, axis=1, keepdims=True)
    c = rng.integers(0, 256, (n, 4), dtype=np.uint8)
    for k in range(nonfinite):
        p[(7 * k + 3) % n, k % 3] = [np.nan, np.inf, MINF][k % 3]
        nrm[(11 * k + 5) % n, (k + 1) % 3] = [MINF, np.nan][k % 2]
    return p, nrm, c


def test_describe_says_what_is_pinned():
    assert "stand-ins" in R.describe()


@pytest.mark.skipif(not os.path.isdir(os.path.join(R.REFERENCE_ROOT, "Data")), reason="the reference's bundled .off files (ICP_REFERENCE_ROOT/Data) are absent")
def test_bunny_fixture_equals_reference_loader(bunny):
    src, tgt, _, _ = bunny
    for cloud, name in ((tgt, "bunny_part1.off"), (src, "bunny_part2_trans.off")):
        p, n = R.cloud_from_off(os.path.join(R.REFERENCE_ROOT, "Data", name))      # SimpleMesh::loadMesh + PointCloud(mesh)
        assert np.array_equal(p, cloud.points)
        assert np.array_equal(n, cloud.normals)


def test_transforms_bit_exact():
    p, n, _ = _cloud(5000, 1, nonfinite=4)
    for s in range(3):
        pose = _pose(s, 0.5, 40.0)
        assert np.array_equal(R.transform_points(pose, p), O.transform_points(pose, p), equal_nan=True)
        assert np.array_equal(R.transform_normals(pose, n), O.transform_normals(pose, n), equal_nan=True)


@pytest.mark.parametrize("quant", [None, 16])
def test_knn3_indices_bit_exact(quant):
    tgt, _, _ = _cloud(3000, 2, quant=quant, nonfinite=3)
    qry, _, _ = _cloud(2000, 3, quant=quant, nonfinite=5)
    for max_d2 in (1e-3, 0.05, 10.0):
        idx, w = R.knn_flann(tgt, qry, max_d2)
        m = O.knn_brute(tgt, qry, max_d2)
        assert np.array_equal(idx, m["idx"]) and np.array_equal(w, m["weight"])
        m2 = O.KdTree(tgt).query(qry, max_d2)
        assert np.array_equal(idx, m2["idx"])
        assert (idx >= 0).any() and (idx < 0).any() or max_d2 == 10.0


def test_flann_stand_in_kdtree_equals_exhaustive_scan():
    tgt, _, tc = _cloud(4000, 21, quant=16, nonfinite=4)
    qry, _, qc = _cloud(3000, 22, quant=16, nonfinite=4)
    try:
        for colours in (False, True):
            a = (tc, qc) if colours else (None, None)
            R.set_flann_exhaustive(True)
            i0, w0 = R.knn_flann(tgt, qry, 0.05, *a)
            R.set_flann_exhaustive(False)
            i1, w1 = R.knn_flann(tgt, qry, 0.05, *a)
            assert np.array_equal(i0, i1) and np.array_equal(w0, w1) and (i0 >= 0).sum() > 300
    finally:
        R.set_flann_exhaustive(False)


def test_knn6_colour_indices_bit_exact():
    tgt, _, tc = _cloud(3000, 4, quant=8)
    qry, _, qc = _cloud(2000, 5, quant=8)
    tc[:, :3] //= 64; qc[:, :3] //= 64          # few colour levels: spatial ties decided by colour
    tc[:, :3] *= 64; qc[:, :3] *= 64
    for max_d2 in (0.02, 10.0):
        idx, w = R.knn_flann(tgt, qry, max_d2, tc, qc)
        m = O.knn_brute(tgt, qry, max_d2, tc, qc)
        assert np.array_equal(idx, m["idx"]) and np.array_equal(w, m["weight"])
        assert np.array_equal(idx, O.KdTree(tgt, tc).query(qry, max_d2, qc)["idx"])
    idx3, _ = R.knn_flann(tgt, qry, 10.0)
    assert (idx3 != idx).any()                  # the colour term really changes the answer


def test_reference_brute_force_has_the_tie_rule_the_oracle_uses():
    # NearestNeighbor.h:81-97: strict '>' => lowest index on ties.  (It compares norm() with the
    # squared threshold, :86,93 -- so only the indices are comparable, with a threshold that lets all pass.)
    tgt, _, _ = _cloud(1500, 6, quant=8)
    qry, _, _ = _cloud(1000, 7, quant=8)
    idx, _ = R.knn_brute(tgt, qry, 1e9)
    m = O.knn_brute(tgt, qry, 1e9)
    same = idx == m["idx"]
    assert same.mean() > 0.995
    # where they differ the two candidates are at the same distance after the sqrt
    d = lambda j: np.sqrt(((qry[~same] - tgt[j]) ** 2).sum(1, dtype=np.float32), dtype=np.float32)
    assert np.allclose(d(idx[~same]), d(m["idx"][~same]), rtol=2e-7)


def test_projective_bit_exact_including_unsigned_wrap():
    from icp_variants_b200 import synth
    w, h = 160, 120
    src, tgt, K, gt = synth.tum_pair(seed=5, width=w, height=h)
    fx, fy, cx, cy = K[0, 0], K[1, 1], K[0, 2], K[1, 2]
    for s, max_d2 in ((0, 0.1), (1, 0.01), (2, 1e-4)):
        pose = gt @ _pose(s, 0.01, 0.5) if s else gt
        q = O.transform_points(pose, src.points)
        idx, wt = R.projective(tgt.points, w, h, fx, fy, cx, cy, q, max_d2)
        m = O.projective(tgt.points, w, h, fx, fy, cx, cy, q, max_d2)
        assert np.array_equal(idx, m["idx"]) and np.array_equal(wt, m["weight"])
        assert (idx >= 0).sum() > (1000 if s == 0 else 50)
    # queries projecting within 12 px of the low borders never match (NearestNeighbor.h:385-386)
    u = np.round(q[:, 0] * fx / q[:, 2] + cx); v = np.round(q[:, 1] * fy / q[:, 2] + cy)
    low = np.isfinite(u) & np.isfinite(v) & ((u < 12) | (v < 12)) & (u >= 0) & (v >= 0)
    assert low.sum() > 100 and (idx[low] < 0).all()


@pytest.mark.parametrize("method", [0, 1, 2, 3])
def test_weights_and_rejection_bit_exact(method):
    sp, sn, sc = _cloud(4000, 8, nonfinite=6)
    tp, tn, tc = _cloud(3000, 9, nonfinite=6)
    max_d2 = 0.02
    m0 = O.knn_brute(tp, sp, max_d2)
    idx, w = R.apply_weights(method, max_d2, sp, sn, sc, tp, tn, tc, m0["idx"], m0["weight"])
    m1 = O.apply_weights(method, max_d2, sp, sn, sc, tp, tn, tc, m0)
    assert np.array_equal(idx, m1["idx"]) and np.array_equal(w, m1["weight"], equal_nan=True)
    if method == 2:
        assert (w[idx >= 0] < 0).any()          # weighting.h:22-25: unclamped dot product
    idx2, w2 = R.prune(sn, tn, idx, w)
    m2 = O.prune(sn, tn, m1)
    assert np.array_equal(idx2, m2["idx"]) and np.array_equal(w2, m2["weight"], equal_nan=True)
    assert ((idx >= 0) & (idx2 < 0)).sum() > 100


def test_rejection_boundary_at_sixty_degrees():
    # ICPOptimizer.h:161,170: float acos against the double threshold => cos == 0.5f is rejected
    ang = np.deg2rad(np.linspace(59.99, 60.01, 2001))
    sn = np.stack([np.cos(ang), np.sin(ang), np.zeros_like(ang)], 1).astype(np.float32)
    sn = np.concatenate([sn, [[0.5, np.sqrt(0.75), 0.0]]]).astype(np.float32)
    tn = np.array([[1.0, 0.0, 0.0]], np.float32)
    idx = np.zeros(len(sn), np.int32); w = np.ones(len(sn), np.float32)
    i_r, _ = R.prune(sn, tn, idx, w)
    m = np.zeros(len(sn), O.MATCH_DTYPE); m["weight"] = 1
    i_o = O.prune(sn, tn, m)["idx"]
    assert np.array_equal(i_r, i_o) and (i_r < 0).any() and (i_r >= 0).any()


@pytest.mark.parametrize("metric", [0, 1, 2])
def test_linear_solvers_within_tolerance(metric):
    rng = np.random.default_rng(10 + metric)
    for n, scale in ((6, 1.0), (500, 1.0), (20000, 10.0)):
        d = (rng.uniform(-1, 1, (n, 3)) * scale).astype(np.float32)
        nt = rng.normal(size=(n, 3)).astype(np.float32); nt /= np.linalg.norm(nt, axis=1, keepdims=True)
        inc = _pose(metric, 0.02 * scale, 1.5)
        s = O.transform_points(np.linalg.inv(inc).astype(np.float32), d) + rng.normal(0, 1e-3, (n, 3)).astype(np.float32)
        ns = (nt + rng.normal(0, 0.05, (n, 3))).astype(np.float32)
        w = rng.uniform(0.2, 1.0, n).astype(np.float32)
        rc_r, pr = R.solve_linear(metric, s, d, ns, nt, w)
        rc_o, po = {0: lambda: O.solve_p2p(s, d, w), 1: lambda: O.solve_p2plane(s, d, nt, w), 2: lambda: O.solve_symmetric(s, d, ns, nt, w)}[metric]()
        assert rc_r == 0 and rc_o == 0
        assert rot_err(pr, po) < ROT_TOL, (n, rot_err(pr, po))
        assert np.abs(pr[:3, 3] - po[:3, 3]).max() < TRANS_TOL * scale, (n, np.abs(pr[:3, 3] - po[:3, 3]).max())
        assert rot_err(po, inc) < 1e-2            # and both recover the increment (small-angle linearisation)


def test_linear_solvers_without_matches():
    # Eigen.h:9 expands ASSERT(a) to `if (!a)` WITHOUT parentheses, so `ASSERT(s.size() > 0 && t.size() > 0 && "..")`
    # (ICPOptimizer.h:668,680,788) only fires for s empty and t non-empty -- never here.  With no matches the
    # reference therefore returns a NaN pose (p2p: 0/0 means), an identity increment (p2plane: empty SVD) or spins
    # in computeMean's ASSERT (symmetric, utils.h:138; made to throw in the test build).  The oracle returns -1 and
    # the product ICP_GPU_E_NO_MATCHES for all three (documented deviation).
    e = np.zeros((0, 3), np.float32)
    w = np.zeros(0, np.float32)
    rc, p = R.solve_linear(0, e, e, e, e, w)
    assert rc == 0 and not np.isfinite(p).all()
    rc, p = R.solve_linear(1, e, e, e, e, w)
    assert rc == 0 and np.array_equal(p, np.eye(4, dtype=np.float32))
    assert R.solve_linear(2, e, e, e, e, w)[0] == -2
    assert O.solve_p2p(e, e, w)[0] == -1 and O.solve_p2plane(e, e, e, w)[0] == -1 and O.solve_symmetric(e, e, e, e, w)[0] == -1


def test_increment_to_matrix_and_functors():
    rng = np.random.default_rng(3)
    for x in (np.zeros(6), np.r_[1e-9, -2e-9, 1e-9, 0.1, 0.2, 0.3], rng.normal(0, 0.3, 6)):
        m = R.increment_to_matrix(x)
        # oracle: LM with zero iterations from x is not exposed; check the matrix against Rodrigues in numpy
        th = np.linalg.norm(x[:3])
        K = np.array([[0, -x[2], x[1]], [x[2], 0, -x[0]], [-x[1], x[0], 0]])
        Rm = np.eye(3) + K if th * th <= np.finfo(float).eps else np.eye(3) + np.sin(th) / th * K + (1 - np.cos(th)) / th ** 2 * K @ K
        assert np.allclose(m[:3, :3], Rm, atol=1e-7) and np.allclose(m[:3, 3], x[3:], atol=1e-7)
        s, d, ns, nt = (rng.normal(size=3).astype(np.float32) for _ in range(4))
        y = Rm @ s + x[3:]
        assert np.allclose(R.residuals(0, x, s, d, ns, nt, 0.7), np.float32(0.1) * np.float64(np.float32(0.7)) * (y - d), atol=1e-12)
        assert np.allclose(R.residuals(1, x, s, d, ns, nt, 0.7), np.float64(np.float32(0.7)) * (nt.astype(np.float64) @ (y - d)), atol=1e-12)
        z = Rm.T @ d
        assert np.allclose(R.residuals(2, x, s, d, ns, nt, 0.7), np.float64(np.float32(0.7)) * ((nt.astype(np.float64) + ns) @ (y - z)), atol=1e-12)


def test_pyramid_levels_bit_exact():
    p, n, c = _cloud(5000, 12, nonfinite=9)
    for f in (1, 2, 8, 64):
        pr, nr, cr = R.coarse_resolution(p, n, c, f)
        i = O.coarse_indices(p, n, f)
        assert np.array_equal(pr, p[i]) and np.array_equal(nr, n[i]) and np.array_equal(cr, c[i])


def test_mt19937_selection_bit_exact():
    n = 3000
    p = np.zeros((n, 3), np.float32); p[:, 0] = np.arange(n)      # the x coordinate is the index
    nrm = np.ones((n, 3), np.float32); c = np.zeros((n, 4), np.uint8)
    for seed, proba, k in ((7, 0.5, 1), (7, 0.5, 3), (123456, 0.01, 2), (0, 0.9, 1)):
        ps, _, n_colors = R.selection(p, nrm, c, proba, seed, k)
        r = O.MT19937().seed(seed)
        keep = None
        for _ in range(k):
            keep = [i for i in range(n) if r.canonical() < proba]
        assert ps[:, 0].astype(np.int64).tolist() == keep
        if k > 1:
            assert n_colors > len(keep)          # selection.h:91-92 never clears m_colors (bug, not replicated)


def test_rmse_bit_exact(bunny):
    src, tgt, gs, gt = bunny
    for s in range(3):
        pose = _pose(s)
        assert R.rmse(pose, src.points[gs], tgt.points[gt]) == O.rmse(pose, src.points[gs], tgt.points[gt])
    assert R.rmse(_pose(1), src.points[:1000], tgt.points[:1000]) == pytest.approx(O.rmse(_pose(1), src.points[:1000], tgt.points[:1000]), rel=1e-6)


def test_depth_to_cloud_equals_reference_constructor():
    from icp_variants_b200 import synth
    w, h = 96, 72
    room = synth.make_room(3)
    depth, _ = synth.render_depth(room, np.array([3.0, 5.0, 1.4]), 10.0, 0.0, w, h, 525.0 * w / 640, 525.0 * w / 640, w / 2 - 0.5, h / 2 - 0.5, seed=3)
    rgba = np.random.default_rng(0).integers(0, 256, (h * w + 1, 4), dtype=np.uint8)
    fx = fy = 525.0 * w / 640; cx, cy = w / 2 - 0.5, h / 2 - 0.5
    for keep, ds in ((True, 1), (False, 1), (False, 8)):
        p, n, c = R.cloud_from_depth(depth, rgba, fx, fy, cx, cy, None, keep, ds, 0.1)
        cl = synth.depth_to_cloud(depth, None, fx, fy, cx, cy, keep_original_size=keep, downsample=ds, max_distance=0.1)
        assert p.shape == cl.points.shape
        assert np.array_equal(p, cl.points) and np.array_equal(n, cl.normals)
        # PointCloud.h:151-152 indexes the RGBX frame with the pixel index (bytes i..i+3), not 4*i
        sel = np.arange(0, h * w, ds)
        if not keep:
            allp = synth.depth_to_cloud(depth, None, fx, fy, cx, cy, keep_original_size=True)
            sel = sel[np.isfinite(allp.points[sel]).all(1) & np.isfinite(allp.normals[sel]).all(1)]
        flat = rgba.reshape(-1)
        assert np.array_equal(c, np.stack([flat[sel + k] for k in range(4)], 1))


BUNNY_VARIANTS = [("base", {}), ("random", dict(selection=1, proba=0.5, seed=7)), ("distance_weights", dict(weighting=1)),
                  ("multires", dict(multires=True))]


@pytest.mark.parametrize("minimizer", [0, 1])
@pytest.mark.parametrize("metric", [0, 1, 2])
@pytest.mark.parametrize("name,kw", BUNNY_VARIANTS)
def test_bunny_variant_matrix_registration(bunny, minimizer, metric, name, kw):
    """The 24 rows of Data/bunny_experiments.csv: {LM, linear} x {p2p, p2plane, symmetric} x
    {baseline, random p=0.5, distance weighting, multires}, 20 iterations, max distance^2 0.0003."""
    src, tgt, gs, gt = bunny
    n, pr, hr = R.estimate_pose(minimizer, metric, src.points, src.normals, src.colors, tgt.points, tgt.normals, tgt.colors,
                                src.points[gs], tgt.points[gt], n_iterations=20, max_distance_sq=0.0003, **kw)
    cfg = O.Config(metric=metric, minimizer=minimizer, n_iterations=20, max_distance_sq=0.0003, **kw)
    rc, po, hist, _ = O.estimate_pose(cfg, src.points, src.normals, src.colors, tgt.points, tgt.normals, tgt.colors)
    assert rc == 0 and n == len(hist) == 20
    assert rot_err(pr, po) < ROT_TOL and np.abs(pr[:3, 3] - po[:3, 3]).max() < TRANS_TOL
    ho = np.array([O.rmse(h, src.points[gs], tgt.points[gt]) for h in hist])
    assert np.abs(hr - ho).max() < 1e-4 and abs(hr[-1] - ho[-1]) < 1e-6
    if minimizer == 1:
        assert np.array_equal(pr, po)            # same LM restatement around the reference's own functors


def test_multires_iteration_count_rule(bunny):
    # ICPOptimizer.h:634-655: runs max(nIterations, levels) iterations
    src, tgt, gs, gt = bunny
    for n_it in (2, 4, 7):
        n, pr, _ = R.estimate_pose(0, 1, src.points, src.normals, src.colors, tgt.points, tgt.normals, tgt.colors,
                                   src.points[gs], tgt.points[gt], n_iterations=n_it, multires=True)
        cfg = O.Config(metric=1, n_iterations=n_it, multires=True)
        rc, po, hist, _ = O.estimate_pose(cfg, src.points, src.normals, src.colors, tgt.points, tgt.normals, tgt.colors)
        assert n == len(hist) == max(n_it, 4)
        assert rot_err(pr, po) < ROT_TOL and np.abs(pr[:3, 3] - po[:3, 3]).max() < TRANS_TOL


@pytest.mark.parametrize("minimizer,metric,weighting", [(0, 1, 0), (0, 2, 2), (1, 2, 3), (0, 0, 3)])
def test_eth_shaped_colour_registration(small_eth_pair, minimizer, metric, weighting):
    """k-NN (3-D and 6-D colour) on an ETH-shaped pair, iteration by iteration."""
    from icp_variants_b200 import synth
    pair = small_eth_pair
    src, tgt = pair[0], pair[1]
    sub = slice(None, None, 3)
    sp, sn = src.points[sub], src.normals[sub]
    tp, tn = tgt.points[sub], tgt.normals[sub]
    sc = synth.procedural_colors(sp); tc = synth.procedural_colors(tp)
    color = weighting == 3
    # Teacher-forced: the reference runs ONE iteration from each pose of the oracle's trajectory.  (Free-running
    # trajectories of the two diverge by ~1e-4 after a few iterations on this sparse pair: a 1e-7 pose difference
    # moves a correspondence across the 0.7 m distance threshold, and one such pair among ~1900 shifts the solution.)
    kw = dict(max_distance_sq=0.5, weighting=weighting, color_icp=color)
    cfg = O.Config(metric=metric, minimizer=minimizer, n_iterations=5, **kw)
    rc, po, hist, _ = O.estimate_pose(cfg, sp, sn, sc, tp, tn, tc)
    assert rc == 0 and len(hist) == 5
    prev = np.eye(4, dtype=np.float32)
    for k in range(5):
        n, pr, _ = R.estimate_pose(minimizer, metric, sp, sn, sc, tp, tn, tc, sp[:4], tp[:4], n_iterations=1, init_pose=prev, **kw)
        assert n == 1
        assert rot_err(pr, hist[k]) < ROT_TOL and np.abs(pr[:3, 3] - hist[k][:3, 3]).max() < TRANS_TOL, (k, rot_err(pr, hist[k]))
        prev = hist[k]
    n, pr, _ = R.estimate_pose(minimizer, metric, sp, sn, sc, tp, tn, tc, sp[:4], tp[:4], n_iterations=5, **kw)
    assert n == 5 and rot_err(pr, po) < 1e-3 and np.abs(pr[:3, 3] - po[:3, 3]).max() < 5e-3


def test_projective_symmetric_registration_tum_shaped():
    from icp_variants_b200 import synth
    w, h = 160, 120
    src, tgt, K, gt = synth.tum_pair(seed=9, width=w, height=h)
    cam = (K[0, 0], K[1, 1], K[0, 2], K[1, 2], w, h)
    for minimizer in (0, 1):
        n, pr, _ = R.estimate_pose(minimizer, 2, src.points, src.normals, src.colors, tgt.points, tgt.normals, tgt.colors,
                                   src.points[:4], tgt.points[:4], n_iterations=6, max_distance_sq=0.1, weighting=2, matching=1,
                                   camera=cam, multires=(minimizer == 1))
        cfg = O.Config(metric=2, minimizer=minimizer, n_iterations=6, max_distance_sq=0.1, weighting=2, matching=1,
                       fx=cam[0], fy=cam[1], cx=cam[2], cy=cam[3], width=w, height=h, multires=(minimizer == 1))
        rc, po, hist, _ = O.estimate_pose(cfg, src.points, src.normals, src.colors, tgt.points, tgt.normals, tgt.colors)
        if minimizer == 0:
            # SURVEY 8a: full-size maps hold finite points with MINF normals; the linear reference turns them into a NaN pose
            # (0 * inf rows).  The oracle / product apply the Ceres path's rule instead (documented deviation).
            # ... after which nothing matches and the next iteration ends in computeMean's ASSERT (-2 in the test build).
            assert n == -2 or not np.isfinite(pr).all() or rot_err(pr, po) < ROT_TOL
            assert rc == 0 and np.isfinite(po).all()
        else:
            assert rc == 0 and n == len(hist)
            assert rot_err(pr, po) < ROT_TOL and np.abs(pr[:3, 3] - po[:3, 3]).max() < TRANS_TOL


def test_oracle_cloud_from_depth_equals_reference_constructor():
    """PointCloud.h:78-165 (SURVEY 8f rank 1): the C oracle against the reference's own constructor."""
    from icp_variants_b200 import synth
    w, h = 96, 72
    fx = fy = 525.0 * w / 640; cx, cy = w / 2 - 0.5, h / 2 - 0.5
    depth, _ = synth.render_depth(synth.make_room(3), np.array([3.0, 5.0, 1.4]), 10.0, 0.0, w, h, fx, fy, cx, cy, seed=3)
    rgbx = np.random.default_rng(0).integers(0, 256, 4 * h * w, dtype=np.uint8)
    for keep, ds, md in ((True, 1, 0.1), (False, 1, 0.1), (False, 8, 0.1), (False, 3, 0.05)):
        pr, nr, cr = R.cloud_from_depth(depth, rgbx, fx, fy, cx, cy, None, keep, ds, md)
        po, no, co = O.cloud_from_depth(depth, rgbx, fx, fy, cx, cy, None, keep, ds, md)
        assert pr.shape == po.shape and len(pr) > 20, (keep, ds, md, len(pr))
        assert np.array_equal(pr, po) and np.array_equal(nr, no) and np.array_equal(cr, co)
    # non-identity depth extrinsics (never used by the reference's drivers): the 4x4 inverse is Eigen's in the reference
    # and an fp64 elimination in the oracle / product, so points agree to rounding only
    E = _pose(4, 0.3, 20.0)
    pr, nr, cr = R.cloud_from_depth(depth, rgbx, fx, fy, cx, cy, E, False, 1, 0.1)
    po, no, co = O.cloud_from_depth(depth, rgbx, fx, fy, cx, cy, E, False, 1, 0.1)
    assert pr.shape == po.shape and np.allclose(pr, po, atol=2e-6) and np.array_equal(nr, no) and np.array_equal(cr, co)


def test_benchmark_error_equals_reference(bunny, small_eth_pair):
    src, tgt, gs, gt = bunny
    for s in range(3):
        pose = _pose(s)
        assert R.benchmark_error(pose, src.points[gs], tgt.points[gt]) == O.benchmark_error(pose, src.points[gs], tgt.points[gt])
    a, b = small_eth_pair[0].points[:3000], small_eth_pair[1].points[:3000]
    assert R.benchmark_error(_pose(1), a, b) == pytest.approx(O.benchmark_error(_pose(1), a, b), rel=1e-9)


def test_pca_normals_equal_reference_constructor(small_eth_pair, bunny):
    """PointCloud(pcl::PointCloud<PointXYZ>::Ptr) (PointCloud.h:41-76): k = 5 normals, colours (255,255,255,1).  PCL is
    absent; the reference constructor runs over the PCL stand-in (exhaustive neighbours, published NormalEstimation
    algorithm), so this pins the constructor's own logic and the oracle's restatement, not PCL's numerics."""
    pts = small_eth_pair[1].points[::2].copy()
    pts[7, 1] = np.nan
    n_r, c_r = R.cloud_from_xyz(pts)
    n_o, _ = O.pca_normals(pts, 5)
    assert np.array_equal(n_r, n_o, equal_nan=True)
    assert (c_r == [255, 255, 255, 1]).all() and np.isnan(n_o[7]).all()
    ok = np.isfinite(n_o).all(1)
    assert np.allclose(np.linalg.norm(n_o[ok], axis=1), 1.0, atol=1e-6)
    assert ((-pts[ok] * n_o[ok]).sum(1) >= -1e-6).all()                # flipped towards the viewpoint (the origin)
    n_b, _ = O.pca_normals(bunny[1].points, 5)
    assert np.array_equal(R.cloud_from_xyz(bunny[1].points)[0], n_b, equal_nan=True)


@pytest.mark.parametrize("setter_order,matcher_d2,weight_d2", [(1, 0.005, 0.002), (2, 0.005, 0.0003)])
def test_matcher_and_weighting_distances_are_separate(bunny, setter_order, matcher_d2, weight_d2):
    """The reference keeps two distances: setMatchingMethod re-creates the matcher with MAX_DISTANCE = 0.005 (ICPOptimizer.h:71-78,
    NearestNeighbor.h:5,35) and leaves ICPOptimizer::maxDistance -- the one WeightingMethod divides by (:220,:528) -- alone.  A driver
    that calls setMatchingMaxDistance BEFORE setMatchingMethod (or never) therefore matches with 0.005 and weights with its own
    value (or 0.0003): the oracle reproduces both through max_distance_sq / weight_max_distance_sq."""
    src, tgt, gs, gt = bunny
    for minimizer, metric in ((0, 1), (0, 2), (1, 1)):
        n, pr, _ = R.estimate_pose(minimizer, metric, src.points, src.normals, src.colors, tgt.points, tgt.normals, tgt.colors,
                                   src.points[gs], tgt.points[gt], n_iterations=5, max_distance_sq=0.002, weighting=1, setter_order=setter_order)
        assert n == 5
        cfg = O.Config(metric=metric, minimizer=minimizer, weighting=1, n_iterations=5, max_distance_sq=matcher_d2, weight_max_distance_sq=weight_d2)
        rc, po, _, _ = O.estimate_pose(cfg, src.points, src.normals, src.colors, tgt.points, tgt.normals, tgt.colors)
        assert rc == 0
        assert rot_err(pr, po) < ROT_TOL and np.abs(pr[:3, 3] - po[:3, 3]).max() < TRANS_TOL
        # and the single-distance configuration is a different registration (the test would not notice a merged field otherwise)
        rc, pm, _, _ = O.estimate_pose(O.Config(metric=metric, minimizer=minimizer, weighting=1, n_iterations=5, max_distance_sq=0.002),
                                       src.points, src.normals, src.colors, tgt.points, tgt.normals, tgt.colors)
        assert rot_err(pm, po) > 10 * ROT_TOL or np.abs(pm[:3, 3] - po[:3, 3]).max() > 10 * TRANS_TOL


def test_reference_brute_force_as_written_norm_threshold():
    """NearestNeighborSearchBruteForce compares (p - m).norm() -- candidates AND the threshold (NearestNeighbor.h:86,93): with the
    same number it keeps a different match set than the squared-distance matchers.  The oracle's restatement of exactly that rule
    (what ICP_GPU_NN_BRUTE_NORM runs on the device) is bit-identical to the reference class, ties of rounded norms included."""
    tgt, _, _ = _cloud(1500, 6, quant=8)
    qry, _, _ = _cloud(1000, 7, quant=8)
    for max_d in (0.05, 0.3, 1e9):
        idx, w = R.knn_brute(tgt, qry, max_d)
        m = O.knn_brute_norm(tgt, qry, max_d)
        assert np.array_equal(idx, m["idx"]) and np.array_equal(w, m["weight"])
    assert (R.knn_brute(tgt, qry, 0.05)[0] < 0).any() and (R.knn_brute(tgt, qry, 0.05)[0] >= 0).any()


def test_oracle_as_ref_answers_like_the_reference(bunny, small_eth_pair):
    """oracle/oracle_as_ref.py -- what the device-vs-reference tests call where this build is absent -- through the same calls
    those tests make, against the reference build, at their tolerances: matching / weighting / rejection, projective, the
    brute-force norm threshold and the depth constructor bit-exact, the functor residuals to 1e-12, the linear solvers and the
    three setter orders to 1e-5 rad / 1e-5 m."""
    from icp_variants_b200 import synth
    from oracle import oracle_as_ref as S
    src, tgt, _ = small_eth_pair
    sc, tc = synth.procedural_colors(src.points), synth.procedural_colors(tgt.points)
    pose = _pose(2, 0.05, 2.0)
    q, qn = S.transform_points(pose, src.points), S.transform_normals(pose, src.normals)
    assert np.array_equal(q, R.transform_points(pose, src.points), equal_nan=True)
    assert np.array_equal(qn, R.transform_normals(pose, src.normals), equal_nan=True)
    for color in (False, True):
        a = (tc, sc) if color else (None, None)
        i0, w0 = R.knn_flann(tgt.points, q, 0.5, *a)
        assert all(np.array_equal(x, y) for x, y in zip(S.knn_flann(tgt.points, q, 0.5, *a), (i0, w0)))
        for method in (0, 1, 2, 3):
            r = R.prune(qn, tgt.normals, *R.apply_weights(method, 0.5, q, qn, sc, tgt.points, tgt.normals, tc, i0, w0))
            s = S.prune(qn, tgt.normals, *S.apply_weights(method, 0.5, q, qn, sc, tgt.points, tgt.normals, tc, i0, w0))
            assert np.array_equal(r[0], s[0]) and np.array_equal(r[1], s[1], equal_nan=True)
    w, h = 160, 120
    ps, pt, K, gt = synth.tum_pair(seed=13, width=w, height=h)
    qp = S.transform_points(gt, ps.points)
    r, s = (M.projective(pt.points, w, h, K[0, 0], K[1, 1], K[0, 2], K[1, 2], qp, 0.1) for M in (R, S))
    fin = np.isfinite(qp).all(1)
    assert np.array_equal(r[0][fin], s[0][fin]) and (r[0] >= 0).sum() > 1000
    bt, _, _ = _cloud(1500, 6, quant=8)
    bq, _, _ = _cloud(1000, 7, quant=8)
    for max_d in (0.05, 0.3):
        assert all(np.array_equal(x, y) for x, y in zip(R.knn_brute(bt, bq, max_d), S.knn_brute(bt, bq, max_d)))
    depth, _ = synth.render_depth(synth.make_room(3), np.array([3.0, 5.0, 1.4]), 10.0, 0.0, 96, 72, 78.75, 78.75, 47.5, 35.5, seed=3)
    rgbx = np.random.default_rng(1).integers(0, 256, 4 * 96 * 72, dtype=np.uint8)
    for keep, ds in ((True, 1), (False, 1), (False, 8)):
        r, s = (M.cloud_from_depth(depth, rgbx, 78.75, 78.75, 47.5, 35.5, None, keep, ds, 0.1) for M in (R, S))
        assert all(np.array_equal(x, y, equal_nan=True) for x, y in zip(r, s))
    keep = i0 >= 0
    s_, d_, ns_, nt_ = q[keep], tgt.points[i0[keep]], qn[keep], tgt.normals[i0[keep]]
    wt = np.random.default_rng(2).uniform(0.2, 1.0, len(s_)).astype(np.float32)
    c0 = d_.mean(0)
    for metric in (0, 1, 2):
        ss, dd = ((s_ - c0).astype(np.float32), (d_ - c0).astype(np.float32)) if metric == 0 else (s_, d_)
        (rc_r, pr), (rc_s, ps_) = R.solve_linear(metric, ss, dd, ns_, nt_, wt), S.solve_linear(metric, ss, dd, ns_, nt_, wt)
        assert rc_r == rc_s == 0 and rot_err(pr, ps_) < ROT_TOL and np.abs(pr[:3, 3] - ps_[:3, 3]).max() < TRANS_TOL
    rng = np.random.default_rng(3)
    for x in (np.zeros(6), np.r_[1e-9, -2e-9, 1e-9, 0.1, 0.2, 0.3], rng.normal(0, 0.3, 6)):
        v = [rng.normal(size=3).astype(np.float32) for _ in range(4)]
        for kind in (0, 1, 2):
            assert np.allclose(S.residuals(kind, x, *v, 0.7), R.residuals(kind, x, *v, 0.7), rtol=0, atol=1e-12)
    bs, bt_, gs, gt_ = bunny
    for order in (0, 1, 2):
        r, s = (M.estimate_pose(0, 1, bs.points, bs.normals, bs.colors, bt_.points, bt_.normals, bt_.colors, bs.points[gs], bt_.points[gt_],
                                n_iterations=5, max_distance_sq=0.002, weighting=1, setter_order=order) for M in (R, S))
        assert r[0] == s[0] == 5 and rot_err(r[1], s[1]) < ROT_TOL and np.abs(r[1][:3, 3] - s[1][:3, 3]).max() < TRANS_TOL
