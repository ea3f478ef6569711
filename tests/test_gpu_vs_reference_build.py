"""The CUDA path (through the icp_gpu_* C ABI) against the reference's OWN code, live: oracle/_ref/libicp_ref.so is the
reference's headers compiled in place (see oracle/ref_driver.cpp for what its stand-ins for Eigen / FLANN / Ceres do and do
not pin).  Where that build is absent the same calls are answered by the oracle (oracle/oracle_as_ref.py), and these tests
then compare the device with the oracle.  The oracle answers each of these calls like the reference build
(tests/test_oracle_vs_reference.py::test_oracle_as_ref_answers_like_the_reference, where the build exists); in every checkout
only the stored reference outputs of tests/golden/reference_outputs.npz (the bunny registrations and one stage set) tie it to the
reference (tests/test_reference_golden.py).

Bit-exact: correspondence indices and weights of NearestNeighborSearchFlann (3-D / 6-D) + WeightingMethod +
pruneCorrespondences, and of NearestNeighborSearchProjective.  One iteration of {Linear,Ceres}ICPOptimizer::estimatePose
from the same pose: 1e-5 rad / 1e-5 m (north_star tolerance)."""
import numpy as np
import pytest

from icp_variants_b200 import capi, synth
from oracle import oracle_as_ref, ref

R = ref if ref.available() else oracle_as_ref

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    c = capi.Context(0)
    yield c
    c.close()


def rot_err(a, b):
    return 2.0 * np.arcsin(min(1.0, np.linalg.norm(a[:3, :3].astype(np.float64) - b[:3, :3]) / (2.0 * np.sqrt(2.0))))


def _poses(k):
    rng = np.random.default_rng(5)
    return [np.eye(4, dtype=np.float32)] + [synth.make_pose(rng.uniform(-0.05, 0.05, 3), rng.uniform(-2, 2, 3)) for _ in range(k)]


@pytest.mark.parametrize("weighting,color", [(0, False), (1, False), (2, False), (3, True)])
@pytest.mark.parametrize("nn", [1, 2], ids=["brute", "grid"])
def test_matching_weighting_rejection_equal_reference_classes(ctx, small_eth_pair, weighting, color, nn):
    src, tgt, _ = small_eth_pair
    sc, tc = synth.procedural_colors(src.points), synth.procedural_colors(tgt.points)
    max_d2 = 0.5
    c = capi.default_config()
    c.nn_algorithm, c.max_distance_sq, c.weighting, c.rejection, c.color_icp = nn, max_d2, weighting, 1, int(color)
    ctx.set_config(c)
    ctx.set_target(tgt.points, tgt.normals, tc)
    ctx.set_source(src.points, src.normals, sc)
    for pose in _poses(2):
        q, qn = R.transform_points(pose, src.points), R.transform_normals(pose, src.normals)      # utils.h:106-133
        i0, w0 = R.knn_flann(tgt.points, q, max_d2, tc if color else None, sc if color else None)   # NearestNeighbor.h:143-303
        i1, w1 = R.apply_weights(weighting, max_d2, q, qn, sc, tgt.points, tgt.normals, tc, i0, w0) # weighting.h:39-99
        i2, w2 = R.prune(qn, tgt.normals, i1, w1)                                                   # ICPOptimizer.h:157-174
        idx, w = ctx.query_matches(pose)
        assert np.array_equal(idx, i2), f"{np.count_nonzero(idx != i2)} of {len(idx)} indices differ"
        ok = idx >= 0
        assert np.array_equal(w[ok], w2[ok])
        assert ok.sum() > 1000


def test_projective_equals_reference_class(ctx):
    w, h = 160, 120
    src, tgt, K, gt = synth.tum_pair(seed=13, width=w, height=h)
    c = capi.default_config()
    c.matching, c.max_distance_sq, c.rejection, c.weighting = 1, 0.1, 0, 0
    ctx.set_config(c); ctx.set_camera(K, w, h)
    ctx.set_target(tgt.points, tgt.normals, tgt.colors)
    ctx.set_source(src.points, src.normals, src.colors)
    for pose in (gt, gt @ _poses(1)[1], np.eye(4, dtype=np.float32)):
        q = R.transform_points(pose, src.points)
        i0, w0 = R.projective(tgt.points, w, h, K[0, 0], K[1, 1], K[0, 2], K[1, 2], q, 0.1)         # NearestNeighbor.h:333-421
        idx, wt = ctx.query_matches(pose)
        fin = np.isfinite(q).all(1)          # a MINF query is skipped by the reference, leaving a value-initialised Match{0, 0.f} (:353)
        assert np.array_equal(idx[fin], i0[fin])
        assert (idx >= 0).sum() > 1000


@pytest.mark.parametrize("minimizer,metric,weighting", [(0, 0, 0), (0, 1, 0), (0, 2, 2), (1, 1, 1), (1, 2, 0)])
def test_one_iteration_equals_reference_estimatePose(ctx, small_eth_pair, minimizer, metric, weighting):
    """Teacher-forced: both run ONE iteration of the loop from the same pose, along the device's own trajectory."""
    src, tgt, _ = small_eth_pair
    sub = slice(None, None, 2)
    sp, sn, tp, tn = src.points[sub], src.normals[sub], tgt.points[sub], tgt.normals[sub]
    sc = np.zeros((len(sp), 4), np.uint8); tc = np.zeros((len(tp), 4), np.uint8)
    c = capi.default_config()
    c.metric, c.minimizer, c.weighting, c.n_iterations, c.max_distance_sq, c.nn_algorithm = metric, minimizer, weighting, 4, 0.5, 2
    ctx.set_config(c)
    ctx.set_target(tp, tn, tc); ctx.set_source(sp, sn, sc)
    pose, hist, n_it = ctx.estimate_pose()
    assert n_it == 4
    prev = np.eye(4, dtype=np.float32)
    for k in range(n_it):
        n, pr, _ = R.estimate_pose(minimizer, metric, sp, sn, sc, tp, tn, tc, sp[:4], tp[:4], n_iterations=1, max_distance_sq=0.5,
                                   weighting=weighting, init_pose=prev)
        assert n == 1
        # metric 0: the reference's Procrustes path accumulates the two means and the 3x3 moment in fp32 over coordinates of up
        # to 17 m (1 ulp = 1.9e-6 m) and forms t = R(mean_d - mean_s) - R mean_d + mean_d in fp32: a few ulps of translation
        # noise of its own, which the fp64 accumulation of the device does not reproduce
        trans_tol = 3e-5 if metric == 0 else 1e-5
        assert rot_err(pr, hist[k]) < 1e-5 and np.abs(pr[:3, 3] - hist[k][:3, 3]).max() < trans_tol, (k, rot_err(pr, hist[k]))
        prev = hist[k]


def test_depth_constructor_equals_reference(ctx):
    w, h = 160, 120
    frames, K, _ = synth.tum_sequence(n_frames=1, seed=4, width=w, height=h)
    rgbx = np.random.default_rng(1).integers(0, 256, 4 * w * h, dtype=np.uint8)
    for keep, ds in ((True, 1), (False, 1), (False, 8)):
        pr, nr, cr = R.cloud_from_depth(frames[0], rgbx, K[0, 0], K[1, 1], K[0, 2], K[1, 2], None, keep, ds, 0.1)   # PointCloud.h:78-165
        pg, ng, cg = ctx.cloud_from_depth(frames[0], rgbx, K, None, keep, ds, 0.1)
        assert np.array_equal(pg, pr, equal_nan=True) and np.array_equal(ng, nr, equal_nan=True) and np.array_equal(cg, cr)


@pytest.mark.parametrize("setter_order", [0, 1, 2])
def test_dropin_setters_keep_matcher_and_weighting_distances_apart(bunny, setter_order):
    """ICPOptimizer drop-in (icp_variants_b200/optimizer.py, mirrored by include/icp_b200/ICPOptimizer.h) driven with the reference's
    setters in three orders against the reference's own classes driven the same way: setMatchingMethod resets only the matcher's
    distance to MAX_DISTANCE (ICPOptimizer.h:71-78), setMatchingMaxDistance sets both (:41-44), WeightingMethod sees
    ICPOptimizer::maxDistance (:220,:528)."""
    from icp_variants_b200.optimizer import LinearICPOptimizer, PointCloud
    src, tgt, gs, gt = bunny
    n, pr, _ = R.estimate_pose(0, 1, src.points, src.normals, src.colors, tgt.points, tgt.normals, tgt.colors, src.points[gs], tgt.points[gt],
                               n_iterations=5, max_distance_sq=0.002, weighting=1, setter_order=setter_order)
    assert n == 5
    opt = LinearICPOptimizer(device=0)
    if setter_order == 1:
        opt.setMatchingMaxDistance(0.002)
    opt.setMatchingMethod(0)
    opt.setMetric(1); opt.setNbOfIterations(5)
    if setter_order == 0:
        opt.setMatchingMaxDistance(0.002)
    opt.setWeightingMethod(1)
    pose = opt.estimatePose(src, tgt, np.eye(4, dtype=np.float32), calculateRMSE=False)
    assert rot_err(pr, pose) < 1e-5 and np.abs(pr[:3, 3] - pose[:3, 3]).max() < 1e-5


def test_brute_force_class_thresholds_the_norm_like_the_reference(ctx):
    """ICP_GPU_NN_BRUTE_NORM = NearestNeighborSearchBruteForce as written (NearestNeighbor.h:81-97): bit-exact against the class."""
    rng = np.random.default_rng(3)
    tgt = (np.round(rng.uniform(-1, 1, (1500, 3)) * 8) / 8).astype(np.float32)      # quantised: many exact ties
    qry = (np.round(rng.uniform(-1, 1, (1000, 3)) * 8) / 8 + 0.01).astype(np.float32)
    c = capi.default_config()
    c.nn_algorithm, c.rejection = 3, 0
    for max_d in (0.05, 0.3):
        c.max_distance_sq = max_d
        ctx.set_config(c)
        ctx.set_target(tgt, None, None); ctx.set_source(qry, None, None)
        idx, w = ctx.query_matches(np.eye(4, dtype=np.float32))
        i0, w0 = R.knn_brute(tgt, qry, max_d)
        assert np.array_equal(idx, i0) and np.array_equal(w, w0)
        assert (idx >= 0).any() and ((idx < 0).any() or max_d > 0.05)


def test_value_level_entry_points_equal_reference_functions(ctx, small_eth_pair):
    """icp_gpu_transform_points / _normals, icp_gpu_apply_weights and icp_gpu_solve_linear -- what the drop-in's transformPoints,
    WeightingMethod, ProcrustesAligner (include/icp_b200/utils.h, weighting.h, ProcrustesAligner.h) call -- against the reference's own
    functions: bit-exact transforms and weights, 1e-5 rad / 1e-5 m for the solvers."""
    src, tgt, _ = small_eth_pair
    sc, tc = synth.procedural_colors(src.points), synth.procedural_colors(tgt.points)
    pose = _poses(1)[1]
    q, qn = ctx.transform_points(pose, src.points), ctx.transform_normals(pose, src.normals)
    assert np.array_equal(q, R.transform_points(pose, src.points), equal_nan=True)                 # utils.h:106-118
    assert np.array_equal(qn, R.transform_normals(pose, src.normals), equal_nan=True)              # utils.h:122-133
    i0, w0 = R.knn_flann(tgt.points, q, 0.5)
    for method in (0, 1, 2, 3):
        _, wr = R.apply_weights(method, 0.5, q, qn, sc, tgt.points, tgt.normals, tc, i0, w0)       # weighting.h:39-99
        wg = ctx.apply_weights(method, 0.5, q, qn, sc, tgt.points, tgt.normals, tc, i0, w0)
        assert np.array_equal(wg, wr)
    keep = i0 >= 0
    s, d, ns, nt = q[keep], tgt.points[i0[keep]], qn[keep], tgt.normals[i0[keep]]
    w = np.random.default_rng(2).uniform(0.2, 1.0, len(s)).astype(np.float32)
    c0 = d.mean(0)
    for metric in (0, 1, 2):
        # metric 0 on centred coordinates: at 17 m the REFERENCE's fp32 Procrustes (means and moments accumulated in fp32) carries
        # 3-4e-5 m of translation noise of its own, which the fp64-accumulating device does not reproduce (DESIGN.md, deviations)
        ss, dd = ((s - c0).astype(np.float32), (d - c0).astype(np.float32)) if metric == 0 else (s, d)
        rc, pr = R.solve_linear(metric, ss, dd, ns, nt, w)                                         # ProcrustesAligner.h / ICPOptimizer.h:676-898
        pg = ctx.solve_linear(metric, ss, dd, ns, nt, w)
        assert rc == 0
        assert rot_err(pr, pg) < 1e-5 and np.abs(pr[:3, 3] - pg[:3, 3]).max() < 1e-5, (metric, rot_err(pr, pg), np.abs(pr[:3, 3] - pg[:3, 3]).max())
    with pytest.raises(capi.IcpGpuError) as e:
        ctx.solve_linear(1, s[:0], d[:0], ns[:0], nt[:0])
    assert e.value.code == capi.E_NO_MATCHES
