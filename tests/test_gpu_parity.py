"""GPU parity tests (run on the B200 box with -m gpu): the CUDA path, called through the icp_gpu_* C
ABI, against the CPU oracle on the same inputs.

Protocol (SURVEY.md section 8c):
  (i)  teacher-forced: at every pose of the oracle's trajectory the device matcher must return the
       oracle's correspondence indices BIT-EXACTLY and the same weights;
  (ii) free-running: the pose after the fixed iteration count must agree with the oracle's within
       ROT_TOL rad / TRANS_TOL m (north_star: 1e-5 / 1e-5).
"""
import time

import numpy as np
import pytest

from icp_variants_b200 import capi, synth
from oracle import oracle as orc

pytestmark = pytest.mark.gpu

ROT_TOL = 1e-5     # rad
TRANS_TOL = 1e-5   # m


def rot_angle(pa, pb):
    # ||Ra - Rb||_F = 2*sqrt(2)*sin(theta/2): well conditioned at small angles, unlike acos((tr-1)/2),
    # which turns the 1e-7 non-orthonormality of an fp32 rotation into a 3e-4 rad "angle"
    d = np.linalg.norm(pa[:3, :3].astype(np.float64) - pb[:3, :3].astype(np.float64))
    return float(2.0 * np.arcsin(min(d / (2.0 * np.sqrt(2.0)), 1.0)))


def pose_close(pa, pb, rot_tol=ROT_TOL, trans_tol=TRANS_TOL):
    return rot_angle(pa, pb) <= rot_tol and float(np.linalg.norm(pa[:3, 3].astype(np.float64) - pb[:3, 3])) <= trans_tol


def gpu_config(ocfg: orc.Config, **kw) -> capi.Config:
    c = capi.default_config()
    c.metric, c.minimizer, c.matching, c.selection = ocfg.metric, ocfg.minimizer, ocfg.matching, ocfg.selection
    c.proba, c.seed, c.weighting, c.rejection = ocfg.proba, ocfg.seed, ocfg.weighting, ocfg.rejection
    c.max_distance_sq, c.color_icp, c.multires = ocfg.max_distance_sq, int(ocfg.color_icp), int(ocfg.multires)
    c.n_iterations, c.lm_max_iterations = ocfg.n_iterations, ocfg.lm_max_iterations
    c.pyramid_mode = ocfg.pyramid_mode
    for k, v in kw.items():
        setattr(c, k, v)
    return c


@pytest.fixture(scope="module")
def ctx():
    c = capi.Context(0)
    yield c
    c.close()


def load(ctx, src, tgt):
    ctx.set_target(tgt.points, tgt.normals, tgt.colors)
    ctx.set_source(src.points, src.normals, src.colors)


def assert_matches_equal(idx, w, om, what=""):
    assert np.array_equal(idx, om["idx"]), f"{what}: {np.count_nonzero(idx != om['idx'])} of {len(idx)} correspondence indices differ"
    assert np.array_equal(w, om["weight"]), f"{what}: max weight diff {np.nanmax(np.abs(w - om['weight']))}"


# ----------------------------------------------------------------------------- (i) teacher-forced
@pytest.mark.parametrize("nn", [1, 2], ids=["brute", "grid"])
@pytest.mark.parametrize("weighting", [0, 1, 2, 3])
@pytest.mark.parametrize("rejection", [1, 0])
def test_bunny_teacher_forced(ctx, bunny, nn, weighting, rejection):
    src, tgt, _, _ = bunny
    ocfg = orc.Config(metric=1, weighting=weighting, rejection=rejection, max_distance_sq=0.0003, n_iterations=8)
    rc, _, hist, _ = orc.estimate_pose(ocfg, src.points, src.normals, src.colors, tgt.points, tgt.normals, tgt.colors)
    assert rc == 0
    load(ctx, src, tgt)
    ctx.set_config(gpu_config(ocfg, nn_algorithm=nn))
    tree = orc.KdTree(tgt.points)
    poses = [np.eye(4, dtype=np.float32)] + list(hist)
    for k, pose in enumerate(poses):
        om = orc.match_pipeline(ocfg, pose, src.points, src.normals, src.colors, tgt.points, tgt.normals, tgt.colors, tree=tree)
        idx, w = ctx.query_matches(pose)
        assert_matches_equal(idx, w, om, f"iteration {k}")
    assert (om["idx"] >= 0).sum() > 500


@pytest.mark.parametrize("max_d2", [0.1, 10.0])
def test_eth_teacher_forced_grid(ctx, small_eth_pair, max_d2, nn=2):
    src, tgt, _ = small_eth_pair
    ocfg = orc.Config(metric=1, max_distance_sq=max_d2, n_iterations=6)
    rc, _, hist, _ = orc.estimate_pose(ocfg, src.points, src.normals, src.colors, tgt.points, tgt.normals, tgt.colors)
    assert rc == 0
    load(ctx, src, tgt)
    ctx.set_config(gpu_config(ocfg, nn_algorithm=nn))
    tree = orc.KdTree(tgt.points)
    for k, pose in enumerate([np.eye(4, dtype=np.float32)] + list(hist)):
        om = orc.match_pipeline(ocfg, pose, src.points, src.normals, src.colors, tgt.points, tgt.normals, tgt.colors, tree=tree)
        idx, w = ctx.query_matches(pose)
        assert_matches_equal(idx, w, om, f"iteration {k}")
    st = ctx.stats()
    assert st.n_queries == len(src) and st.n_distance_evals > 0


def test_grid_equals_brute_on_ties_and_nonfinite(ctx):
    """Quantised coordinates (many exact ties), duplicated target points, non-finite targets and
    queries: lowest original index must win, non-finite points never match."""
    rng = np.random.default_rng(7)
    tgt = (rng.integers(0, 12, size=(6000, 3)) * 0.25).astype(np.float32)
    tgt[100:200] = tgt[0:100]                      # duplicates with higher indices
    tgt[300] = [np.inf, 0, 0]
    tgt[301] = [np.nan, 1, 1]
    tgt[302] = [-np.inf, -np.inf, -np.inf]
    qry = (rng.integers(-2, 14, size=(4000, 3)) * 0.25 + 0.125 * rng.integers(0, 2, size=(4000, 3))).astype(np.float32)
    qry[5] = [np.nan, 0, 0]
    qry[6] = [-np.inf, -np.inf, -np.inf]
    zeros_t, zeros_q = np.zeros_like(tgt), np.zeros_like(qry)
    ref = orc.knn_brute(tgt, qry, 1.0)
    for nn in (1, 2):
        c = capi.default_config()
        c.nn_algorithm, c.max_distance_sq, c.rejection = nn, 1.0, 0
        ctx.set_config(c)
        ctx.set_target(tgt, zeros_t, None)
        ctx.set_source(qry, zeros_q, None)
        idx, w = ctx.query_matches(np.eye(4, dtype=np.float32))
        assert_matches_equal(idx, w, ref, f"nn={nn}")
    assert ref["idx"][5] == -1 and ref["idx"][6] == -1


def test_color_icp_6d_teacher_forced(ctx):
    src, tgt, _ = synth.eth_pair(seed=4321, n_sweeps=40, n_beams=120, colors="texture")
    ocfg = orc.Config(metric=2, weighting=3, color_icp=True, max_distance_sq=0.1, n_iterations=3)
    rc, _, hist, _ = orc.estimate_pose(ocfg, src.points, src.normals, src.colors, tgt.points, tgt.normals, tgt.colors)
    assert rc == 0
    load(ctx, src, tgt)
    tree = orc.KdTree(tgt.points, tgt.colors)
    for nn in (1, 2):
        ctx.set_config(gpu_config(ocfg, nn_algorithm=nn))
        for k, pose in enumerate([np.eye(4, dtype=np.float32)] + list(hist)):
            om = orc.match_pipeline(ocfg, pose, src.points, src.normals, src.colors, tgt.points, tgt.normals, tgt.colors, tree=tree)
            idx, w = ctx.query_matches(pose)
            assert_matches_equal(idx, w, om, f"nn={nn} iteration {k}")


@pytest.fixture(scope="module")
def small_tum():
    return synth.tum_pair(seed=1234, frame_gap=10, width=160, height=120)


@pytest.mark.parametrize("weighting", [0, 2])
def test_projective_teacher_forced(ctx, small_tum, weighting):
    src, tgt, k, _ = small_tum
    ocfg = orc.Config(metric=2, matching=1, weighting=weighting, max_distance_sq=0.1, n_iterations=4,
                      fx=float(k[0, 0]), fy=float(k[1, 1]), cx=float(k[0, 2]), cy=float(k[1, 2]), width=160, height=120)
    rc, _, hist, _ = orc.estimate_pose(ocfg, src.points, src.normals, src.colors, tgt.points, tgt.normals, tgt.colors)
    assert rc == 0
    load(ctx, src, tgt)
    ctx.set_camera(k, 160, 120)
    ctx.set_config(gpu_config(ocfg))
    for it, pose in enumerate([np.eye(4, dtype=np.float32)] + list(hist)):
        om = orc.match_pipeline(ocfg, pose, src.points, src.normals, src.colors, tgt.points, tgt.normals, tgt.colors)
        idx, w = ctx.query_matches(pose)
        assert_matches_equal(idx, w, om, f"iteration {it}")
    assert (om["idx"] > 0).sum() > 1000


def test_selection_subset_query(ctx, bunny):
    src, tgt, _, _ = bunny
    ocfg = orc.Config(metric=0, max_distance_sq=0.0003)
    load(ctx, src, tgt)
    ctx.set_config(gpu_config(ocfg))
    sel = np.arange(3, len(src), 7, dtype=np.int32)
    om = orc.match_pipeline(ocfg, np.eye(4, dtype=np.float32), src.points, src.normals, src.colors, tgt.points, tgt.normals, tgt.colors,
                            sel_idx=sel)
    idx, w = ctx.query_matches(np.eye(4, dtype=np.float32), sel)
    assert_matches_equal(idx, w, om)


# ----------------------------------------------------------------------------- (ii) free-running
VARIANTS = [(mini, metric) for mini in (0, 1) for metric in (0, 1, 2)]


@pytest.mark.parametrize("minimizer,metric", VARIANTS)
@pytest.mark.parametrize("use_graph", [1, 0])
def test_bunny_free_running(ctx, bunny, minimizer, metric, use_graph):
    src, tgt, gs, gt = bunny
    ocfg = orc.Config(metric=metric, minimizer=minimizer, max_distance_sq=0.0003, n_iterations=20)
    rc, opose, ohist, nq = orc.estimate_pose(ocfg, src.points, src.normals, src.colors, tgt.points, tgt.normals, tgt.colors)
    assert rc == 0
    load(ctx, src, tgt)
    ctx.set_config(gpu_config(ocfg, use_graph=use_graph))
    pose, hist, n_it = ctx.estimate_pose()
    assert n_it == 20 and len(hist) == 20
    assert ctx.stats().n_queries == nq
    for k in range(20):
        assert pose_close(hist[k], ohist[k]), f"iteration {k}: rot {rot_angle(hist[k], ohist[k]):.2e} trans {np.linalg.norm(hist[k][:3, 3] - ohist[k][:3, 3]):.2e}"
    assert pose_close(pose, opose)
    assert np.array_equal(pose, hist[-1])
    # running it again replays the cached graph and must give the same bits
    pose2, _, _ = ctx.estimate_pose()
    assert np.array_equal(pose, pose2)


@pytest.mark.parametrize("minimizer,metric", VARIANTS)
def test_eth_free_running(ctx, small_eth_pair, minimizer, metric):
    """Tiled grid search with warm starts from the previous iteration's neighbours."""
    src, tgt, _ = small_eth_pair
    ocfg = orc.Config(metric=metric, minimizer=minimizer, max_distance_sq=0.1, n_iterations=10)
    rc, opose, ohist, _ = orc.estimate_pose(ocfg, src.points, src.normals, src.colors, tgt.points, tgt.normals, tgt.colors)
    assert rc == 0
    load(ctx, src, tgt)
    ctx.set_config(gpu_config(ocfg))
    pose, hist, n_it = ctx.estimate_pose()
    assert n_it == 10
    assert pose_close(pose, opose), f"rot {rot_angle(pose, opose):.2e} trans {np.linalg.norm(pose[:3, 3] - opose[:3, 3]):.2e}"


@pytest.mark.parametrize("weighting", [1, 2])
def test_bunny_weighted_free_running(ctx, bunny, weighting):
    src, tgt, _, _ = bunny
    ocfg = orc.Config(metric=1, weighting=weighting, max_distance_sq=0.0003, n_iterations=20)
    rc, opose, _, _ = orc.estimate_pose(ocfg, src.points, src.normals, src.colors, tgt.points, tgt.normals, tgt.colors)
    load(ctx, src, tgt)
    ctx.set_config(gpu_config(ocfg))
    pose, _, _ = ctx.estimate_pose()
    assert pose_close(pose, opose)


@pytest.mark.parametrize("minimizer,metric", [(0, 1), (0, 2), (1, 2)])
def test_bunny_multires(ctx, bunny, minimizer, metric):
    """Stride pyramid (PointCloud.h:325-343, ICPOptimizer.h:503-525,634-655): 1054 points -> strides 8,4,2,1."""
    src, tgt, _, _ = bunny
    ocfg = orc.Config(metric=metric, minimizer=minimizer, multires=True, max_distance_sq=0.0003, n_iterations=20)
    rc, opose, ohist, nq = orc.estimate_pose(ocfg, src.points, src.normals, src.colors, tgt.points, tgt.normals, tgt.colors)
    assert rc == 0
    load(ctx, src, tgt)
    ctx.set_config(gpu_config(ocfg))
    assert ctx.max_iterations() == 20
    pose, hist, n_it = ctx.estimate_pose()
    assert n_it == len(ohist)
    assert ctx.stats().n_queries == nq
    assert pose_close(pose, opose)


@pytest.mark.parametrize("minimizer,metric", [(0, 1), (0, 2), (1, 1)])
def test_voxel_pyramid(ctx, small_eth_pair, minimizer, metric):
    """ICP_GPU_PYRAMID_VOXEL (extension): levels = one point per occupied source-grid cell; the oracle restates the
    device grid operation by operation, so level membership -- and hence query counts and poses -- must agree."""
    src, tgt, _ = small_eth_pair
    src = synth.Cloud(src.points.copy(), src.normals.copy(), src.colors.copy())
    src.normals[5::97] = np.nan                     # invalid normals are never level representatives
    src.points[11::501] = -np.inf
    ocfg = orc.Config(metric=metric, minimizer=minimizer, multires=True, pyramid_mode=1, max_distance_sq=0.1, n_iterations=10)
    rc, opose, ohist, nq = orc.estimate_pose(ocfg, src.points, src.normals, src.colors, tgt.points, tgt.normals, tgt.colors)
    assert rc == 0
    load(ctx, src, tgt)
    ctx.set_config(gpu_config(ocfg, nn_algorithm=2))
    pose, hist, n_it = ctx.estimate_pose()
    assert n_it == len(ohist)
    assert ctx.stats().n_queries == nq
    assert pose_close(pose, opose), f"rot {rot_angle(pose, opose):.2e} trans {np.linalg.norm(pose[:3, 3] - opose[:3, 3]):.2e}"
    cfg = gpu_config(ocfg, nn_algorithm=2, selection=1, proba=0.5, selection_rng=0)
    with pytest.raises(capi.IcpGpuError) as e:      # host-drawn masks cannot follow device-built levels
        ctx.set_config(cfg)
    assert e.value.code == capi.E_ARG


def test_multires_more_levels_than_iterations(ctx, small_eth_pair):
    src, tgt, _ = small_eth_pair
    ocfg = orc.Config(metric=1, multires=True, max_distance_sq=0.1, n_iterations=3)
    rc, opose, ohist, nq = orc.estimate_pose(ocfg, src.points, src.normals, src.colors, tgt.points, tgt.normals, tgt.colors)
    assert rc == 0 and len(ohist) > 3
    load(ctx, src, tgt)
    ctx.set_config(gpu_config(ocfg))
    assert ctx.max_iterations() == len(ohist)
    pose, hist, n_it = ctx.estimate_pose()
    assert n_it == len(ohist) and ctx.stats().n_queries == nq
    assert pose_close(pose, opose)


@pytest.mark.parametrize("multires", [False, True])
def test_random_selection_mt19937(ctx, bunny, multires):
    """selection.h:88-104 with an explicit seed: the host draws the reference's mt19937 stream."""
    src, tgt, _, _ = bunny
    ocfg = orc.Config(metric=1, selection=1, proba=0.5, seed=42, multires=multires, max_distance_sq=0.0003, n_iterations=12)
    rc, opose, ohist, nq = orc.estimate_pose(ocfg, src.points, src.normals, src.colors, tgt.points, tgt.normals, tgt.colors)
    assert rc == 0
    load(ctx, src, tgt)
    ctx.set_config(gpu_config(ocfg))
    pose, hist, n_it = ctx.estimate_pose()
    assert n_it == len(ohist) and ctx.stats().n_queries == nq
    assert pose_close(pose, opose)


def test_random_selection_device_stream(ctx, bunny):
    """The device selection stream is not reference-compatible; it must select ~p of the points and converge."""
    src, tgt, gs, gt = bunny
    c = capi.default_config()
    c.metric, c.selection, c.proba, c.seed, c.selection_rng, c.n_iterations = 2, 1, 0.5, 3, 1, 20
    load(ctx, src, tgt)
    ctx.set_config(c)
    pose, _, n_it = ctx.estimate_pose()
    frac = ctx.stats().n_queries / (20 * len(src))
    assert 0.45 < frac < 0.55
    assert orc.rmse(pose, src.points[gs], tgt.points[gt]) < 1e-3


def test_projective_free_running(ctx, small_tum):
    src, tgt, k, gt = small_tum
    ocfg = orc.Config(metric=2, matching=1, weighting=2, max_distance_sq=0.1, n_iterations=10,
                      fx=float(k[0, 0]), fy=float(k[1, 1]), cx=float(k[0, 2]), cy=float(k[1, 2]), width=160, height=120)
    rc, opose, _, _ = orc.estimate_pose(ocfg, src.points, src.normals, src.colors, tgt.points, tgt.normals, tgt.colors)
    assert rc == 0
    load(ctx, src, tgt)
    ctx.set_camera(k, 160, 120)
    ctx.set_config(gpu_config(ocfg))
    pose, _, n_it = ctx.estimate_pose()
    assert n_it == 10
    assert pose_close(pose, opose), f"rot {rot_angle(pose, opose):.2e} trans {np.linalg.norm(pose[:3, 3] - opose[:3, 3]):.2e}"


@pytest.mark.parametrize("metric,weighting,multires", [(0, 0, False), (1, 1, False), (2, 2, False), (1, 3, True), (2, 0, True)])
def test_fused_reduction_equals_match_records(ctx, small_eth_pair, metric, weighting, multires):
    """collect_stats = 0 lets the linear minimiser evaluate weighting + rejection inside the reduction instead of reading
    match records: same arithmetic, so the poses must be bit-identical to the unfused path."""
    src, tgt, _ = small_eth_pair
    c = capi.default_config()
    c.metric, c.weighting, c.multires, c.max_distance_sq, c.n_iterations, c.nn_algorithm = metric, weighting, int(multires), 0.1, 8, 2
    c.selection, c.proba, c.selection_rng, c.seed = 1, 0.7, 1, 5
    load(ctx, src, tgt)
    poses = []
    for stats in (1, 0):
        c.collect_stats = stats
        ctx.set_config(c)
        pose, hist, _ = ctx.estimate_pose()
        poses.append(hist)
    assert np.array_equal(poses[0], poses[1])


def test_bunny_known_answer(ctx, bunny):
    """SURVEY.md section 4: bunny_part2_trans maps onto bunny_part1 by Rz(12.2348 deg), t=(-0.0151362,-0.0032822,0)."""
    src, tgt, gs, gt = bunny
    c = capi.default_config()
    c.metric, c.n_iterations = 2, 20
    load(ctx, src, tgt)
    ctx.set_config(c)
    pose, _, _ = ctx.estimate_pose()
    assert abs(np.degrees(np.arctan2(pose[1, 0], pose[0, 0])) - 12.2348) < 0.1
    assert np.allclose(pose[:3, 3], [-0.0151362, -0.0032822, 0.0], atol=3e-4)
    assert orc.rmse(pose, src.points[gs], tgt.points[gt]) < 4e-4


# ----------------------------------------------------------------------------- error behaviour
def test_error_codes(bunny):
    src, tgt, _, _ = bunny
    with capi.Context(0) as c:
        with pytest.raises(capi.IcpGpuError) as e:
            c.estimate_pose()
        assert e.value.code == capi.E_STATE
        c.set_target(tgt.points, tgt.normals, tgt.colors)
        far = src.points + np.float32(100.0)
        c.set_source(far, src.normals, src.colors)
        with pytest.raises(capi.IcpGpuError) as e:      # the reference hangs in ASSERT (Eigen.h:9)
            c.estimate_pose()
        assert e.value.code == capi.E_NO_MATCHES
        assert np.array_equal(e.value.pose, np.eye(4, dtype=np.float32))
        cfg = capi.default_config()
        cfg.matching = 1
        c.set_config(cfg)
        with pytest.raises(capi.IcpGpuError) as e:      # projective without camera
            c.estimate_pose()
        assert e.value.code == capi.E_STATE
        cfg.metric = 7
        with pytest.raises(capi.IcpGpuError) as e:
            c.set_config(cfg)
        assert e.value.code == capi.E_ARG


def test_empty_clouds(ctx, bunny):
    src, tgt, _, _ = bunny
    c = capi.default_config()
    ctx.set_config(c)
    ctx.set_target(np.zeros((0, 3), np.float32), np.zeros((0, 3), np.float32), None)
    ctx.set_source(src.points, src.normals, src.colors)
    idx, w = ctx.query_matches(np.eye(4, dtype=np.float32))
    assert (idx == -1).all() and (w == 0).all()
    ctx.set_target(tgt.points, tgt.normals, tgt.colors)
    ctx.set_source(np.zeros((0, 3), np.float32), np.zeros((0, 3), np.float32), None)
    idx, w = ctx.query_matches(np.eye(4, dtype=np.float32))
    assert len(idx) == 0
    with pytest.raises(capi.IcpGpuError) as e:
        ctx.estimate_pose()
    assert e.value.code == capi.E_NO_MATCHES


# ----------------------------------------------------------------------------- point-sharded iteration (one GPU, two contexts)
@pytest.mark.parametrize("metric", [0, 1, 2])
def test_point_sharded_equals_single(bunny, metric):
    """Two contexts each hold the whole target and half of the source; summing their partial rows and
    applying the sum on both must reproduce the single-context trajectory."""
    src, tgt, _, _ = bunny
    cfg = capi.default_config()
    cfg.metric, cfg.n_iterations = metric, 5
    with capi.Context(0) as full, capi.Context(0) as a, capi.Context(0) as b:
        full.set_config(cfg); a.set_config(cfg); b.set_config(cfg)
        full.set_target(tgt.points, tgt.normals, tgt.colors)
        full.set_source(src.points, src.normals, src.colors)
        ref_pose, _, _ = full.estimate_pose()
        h = len(src) // 2
        for c, sl in ((a, slice(0, h)), (b, slice(h, None))):
            c.set_target(tgt.points, tgt.normals, tgt.colors)
            c.set_source(src.points[sl], src.normals[sl], src.colors[sl])
        eye = np.eye(4, dtype=np.float32)
        a.iteration_begin(eye); b.iteration_begin(eye)
        for _ in range(5):
            for ph in range(a.iteration_phases()):
                tot = a.iteration_local(ph) + b.iteration_local(ph)
                a.iteration_apply(ph, tot); b.iteration_apply(ph, tot)
        pa, pb = a.iteration_end(), b.iteration_end()
        assert np.array_equal(pa, pb)
        assert pose_close(pa, ref_pose, 1e-6, 1e-6)


# ----------------------------------------------------------------------------- the same with the exchange inside the reduction kernel
def _peer_pair(tgt, src, cfg, n_ctx=2):
    """n contexts on this GPU, each with the whole target and a contiguous shard of the source, mailboxes attached."""
    from icp_variants_b200 import parallel
    ctxs = [capi.Context(0) for _ in range(n_ctx)]
    for r, c in enumerate(ctxs):
        sl = parallel.shard_points(len(src), n_ctx, r)
        c.set_config(cfg)
        c.set_target(tgt.points, tgt.normals, tgt.colors)
        c.set_source(src.points[sl], src.normals[sl], src.colors[sl])
    addr = [c.peer_address() for c in ctxs]              # every mailbox exists (zeroed) before anybody attaches
    for r, c in enumerate(ctxs):
        c.peer_attach_ptrs(r, n_ctx, addr)
    return ctxs


@pytest.mark.parametrize("metric,minimizer,n_ctx,graph", [(0, 0, 2, 1), (1, 0, 2, 1), (2, 0, 2, 1), (1, 0, 3, 1), (1, 0, 2, 0), (1, 1, 2, 1), (2, 1, 2, 1)])
def test_peer_memory_sharded_registration_equals_single(bunny, monkeypatch, metric, minimizer, n_ctx, graph):
    """icp_gpu_peer_*: the last block of every reduction stores its row into the peers' mailboxes and sums the rows
    it receives, so each context's ordinary estimate_pose runs the point-sharded registration without the host.
    All contexts must end with the bit-identical pose, equal to the single-context one within the pose tolerance."""
    monkeypatch.setenv("ICP_GPU_PEER_TIMEOUT_MS", "20000")
    src, tgt, _, _ = bunny
    cfg = capi.default_config()
    cfg.metric, cfg.minimizer, cfg.n_iterations, cfg.use_graph, cfg.collect_stats = metric, minimizer, 5, graph, 0
    with capi.Context(0) as full:
        full.set_config(cfg)
        full.set_target(tgt.points, tgt.normals, tgt.colors)
        full.set_source(src.points, src.normals, src.colors)
        ref_pose, _, _ = full.estimate_pose()
    ctxs = _peer_pair(tgt, src, cfg, n_ctx)
    try:
        for rep in range(2):                              # twice: the exchange counter runs on across registrations
            for c in ctxs:
                c.estimate_pose_async()                   # enqueue only: the kernels of the contexts wait for each other
            poses = [c.estimate_pose_finish()[0] for c in ctxs]
            for q in poses[1:]:
                assert np.array_equal(poses[0], q)
            assert pose_close(poses[0], ref_pose, 1e-6, 1e-6)
        ctxs[0].peer_detach()                             # detached: a single-context registration of its own shard again
        alone, _, _ = ctxs[0].estimate_pose()
        assert np.isfinite(alone).all()
    finally:
        for c in ctxs:
            c.close()


def test_peer_memory_sharded_grid_search_fused_reduction(small_eth_pair, monkeypatch):
    """The same on the BVH search path, where the reduction evaluates weighting / rejection itself (fused stages 3-4):
    10 point-to-plane iterations of an ETH-shaped pair split over two contexts."""
    monkeypatch.setenv("ICP_GPU_PEER_TIMEOUT_MS", "20000")
    src, tgt, _ = small_eth_pair
    cfg = capi.default_config()
    cfg.metric, cfg.n_iterations, cfg.max_distance_sq, cfg.nn_algorithm, cfg.collect_stats = 1, 10, 10.0, 2, 0
    with capi.Context(0) as full:
        full.set_config(cfg)
        full.set_target(tgt.points, tgt.normals, tgt.colors)
        full.set_source(src.points, src.normals, src.colors)
        ref_pose, _, _ = full.estimate_pose()
    ctxs = _peer_pair(tgt, src, cfg, 2)
    try:
        for c in ctxs:
            c.estimate_pose_async()
        (pa, na), (pb, nb) = [c.estimate_pose_finish() for c in ctxs]
        assert na == nb == 10 and np.array_equal(pa, pb)
        assert pose_close(pa, ref_pose, 1e-6, 1e-6)
    finally:
        for c in ctxs:
            c.close()


def test_peer_memory_missing_peer_times_out_with_an_error(bunny, monkeypatch):
    """A rank whose peer never arrives must finish with ICP_GPU_E_PEER, not hang the GPU."""
    monkeypatch.setenv("ICP_GPU_PEER_TIMEOUT_MS", "50")
    src, tgt, _, _ = bunny
    cfg = capi.default_config()
    cfg.metric, cfg.n_iterations = 1, 2
    ctxs = _peer_pair(tgt, src, cfg, 2)
    try:
        with pytest.raises(capi.IcpGpuError) as e:
            ctxs[0].estimate_pose()                       # rank 1 never runs
        assert e.value.code == capi.E_PEER
        with pytest.raises(capi.IcpGpuError):             # the NCCL-style split iteration is refused while peers are attached
            ctxs[1].iteration_begin(np.eye(4, dtype=np.float32))
        # The rank that gave up poisoned the exchange: the late peer must fail too -- at once, not after its own time-out, and
        # not "succeed" on the stale rows rank 0 left in its mailbox.
        monkeypatch.setenv("ICP_GPU_PEER_TIMEOUT_MS", "20000")
        t0 = time.perf_counter()
        with pytest.raises(capi.IcpGpuError) as e:
            ctxs[1].estimate_pose()
        assert e.value.code == capi.E_PEER and time.perf_counter() - t0 < 5.0
    finally:
        for c in ctxs:
            c.close()


def test_peer_memory_lost_peer_costs_one_timeout_per_registration(bunny, monkeypatch):
    """Once a rank has raised ICP_GPU_E_PEER the remaining launches of its registration skip the exchange: 8 iterations of the
    symmetric metric (16 exchanges) with a 300 ms time-out take about one time-out, not sixteen."""
    monkeypatch.setenv("ICP_GPU_PEER_TIMEOUT_MS", "300")
    src, tgt, _, _ = bunny
    cfg = capi.default_config()
    cfg.metric, cfg.n_iterations = 2, 8
    ctxs = _peer_pair(tgt, src, cfg, 2)
    try:
        t0 = time.perf_counter()
        with pytest.raises(capi.IcpGpuError) as e:
            ctxs[0].estimate_pose()
        assert e.value.code == capi.E_PEER
        assert time.perf_counter() - t0 < 2.0
    finally:
        for c in ctxs:
            c.close()


def test_peer_memory_ranks_must_plan_the_same_registration(bunny, monkeypatch):
    """Ranks whose iteration counts differ would wait for exchanges that never come: the first exchange compares the plans
    and every rank finishes with ICP_GPU_E_PEER; the multi-resolution schedule (derived from the local shard) is refused."""
    monkeypatch.setenv("ICP_GPU_PEER_TIMEOUT_MS", "20000")
    src, tgt, _, _ = bunny
    cfg = capi.default_config()
    cfg.metric, cfg.n_iterations = 1, 4
    ctxs = _peer_pair(tgt, src, cfg, 2)
    try:
        cfg.n_iterations = 6
        ctxs[1].set_config(cfg)
        t0 = time.perf_counter()
        for c in ctxs:
            c.estimate_pose_async()
        for c in ctxs:
            with pytest.raises(capi.IcpGpuError) as e:
                c.estimate_pose_finish()
            assert e.value.code == capi.E_PEER
        assert time.perf_counter() - t0 < 10.0
        cfg.multires = 1
        ctxs[0].set_config(cfg)
        with pytest.raises(capi.IcpGpuError) as e:
            ctxs[0].estimate_pose()
        assert e.value.code == capi.E_ARG
    finally:
        for c in ctxs:
            c.close()


# ----------------------------------------------------------------------------- BASELINE.json full sizes
@pytest.fixture(scope="module")
def full_eth_pair():
    """configs[1]: 344 sweeps x 1077 beams = 370 488 points per scan."""
    return synth.eth_pair(seed=1234)


def test_full_size_eth_correspondences_bit_exact(ctx, full_eth_pair):
    """At the benchmark's size the device search must still return exactly the oracle's (kd-tree, == brute force)
    correspondences, at the start pose and -- warm-started from its own previous answer -- at a later pose."""
    src, tgt, _ = full_eth_pair
    assert len(src) == 370488 and len(tgt) == 370488
    ocfg = orc.Config(metric=1, max_distance_sq=10.0)
    load(ctx, src, tgt)
    ctx.set_config(gpu_config(ocfg, nn_algorithm=2))
    tree = orc.KdTree(tgt.points)
    later = synth.make_pose([-0.02, -0.015, -0.004], [-0.15, -0.08, -0.4])
    for pose in (np.eye(4, dtype=np.float32), later, np.eye(4, dtype=np.float32)):
        om = orc.match_pipeline(ocfg, pose, src.points, src.normals, src.colors, tgt.points, tgt.normals, tgt.colors, tree=tree)
        idx, w = ctx.query_matches(pose)
        assert_matches_equal(idx, w, om)
    assert (om["idx"] >= 0).mean() > 0.5


def test_full_size_eth_registration(ctx, full_eth_pair):
    """The benchmark's registration at full size: the pose after 10 iterations agrees with the oracle's within the
    tolerance, repeating it gives the same bits (deterministic reductions, graph replay), and the graph and
    launch-by-launch paths agree."""
    src, tgt, pert = full_eth_pair
    ocfg = orc.Config(metric=1, max_distance_sq=10.0, n_iterations=10)
    rc, opose, _, nq = orc.estimate_pose(ocfg, src.points, src.normals, src.colors, tgt.points, tgt.normals, tgt.colors)
    assert rc == 0
    load(ctx, src, tgt)
    cfg = gpu_config(ocfg, nn_algorithm=2)
    ctx.set_config(cfg)
    pose, hist, n_it = ctx.estimate_pose()
    assert n_it == 10 and ctx.stats().n_queries == nq
    assert pose_close(pose, opose), f"rot {rot_angle(pose, opose):.2e} trans {np.linalg.norm(pose[:3, 3] - opose[:3, 3]):.2e}"
    # the registration moves the source back towards the frame the perturbation took it from
    before = np.linalg.norm(pert[:3, 3])
    after = np.linalg.norm((pose.astype(np.float64) @ pert.astype(np.float64))[:3, 3])
    assert after < before * 3.5      # (biased by the ~18 % of points without a counterpart; the oracle shows the same)
    pose2, _, _ = ctx.estimate_pose()
    assert np.array_equal(pose, pose2)
    cfg.use_graph = 0
    ctx.set_config(cfg)
    pose3, _, _ = ctx.estimate_pose()
    assert np.array_equal(pose, pose3)


def test_bench_config_as_run_370k_30_iterations(ctx, full_eth_pair):
    """BASELINE configs[1] exactly as bench.py runs it -- 370 488 x 370 488 points, k-NN, point-to-plane linear, 30 iterations, max
    distance^2 10, rejection on, work counters off (so the fused reduction path) -- against the oracle's free-running loop."""
    src, tgt, _ = full_eth_pair
    ocfg = orc.Config(metric=1, max_distance_sq=10.0, n_iterations=30)
    rc, opose, ohist, _ = orc.estimate_pose(ocfg, src.points, src.normals, src.colors, tgt.points, tgt.normals, tgt.colors)
    assert rc == 0
    load(ctx, src, tgt)
    ctx.set_config(gpu_config(ocfg, nn_algorithm=2, collect_stats=0))
    pose, hist, n_it = ctx.estimate_pose()
    assert n_it == 30
    worst = max(rot_angle(hist[k], ohist[k]) for k in range(30)), max(float(np.linalg.norm(hist[k][:3, 3] - ohist[k][:3, 3])) for k in range(30))
    assert pose_close(pose, opose), f"rot {rot_angle(pose, opose):.2e} trans {np.linalg.norm(pose[:3, 3] - opose[:3, 3]):.2e}"
    assert worst[0] <= ROT_TOL and worst[1] <= TRANS_TOL, worst        # every iteration of the trajectory, not only the last


def test_chunk_chains_graph_and_group_search_change_no_bit(full_eth_pair, monkeypatch):
    """How the search is scheduled is invisible in the results: one, two or three {prep, walk} chunk chains per iteration
    (ICP_GPU_MATCH_CHUNKS; two is the default from 131 072 queries on), launched one by one or as a graph, and runs of deferred
    neighbours searched with one shared descent or each by its own walk (ICP_GPU_GROUP_MIN: 0 = off, 1 = every run) give the same
    trajectory and the same correspondences bit for bit.  The variables are read when a registration is enqueued; a fresh context
    per variant keeps the graph caches apart."""
    src, tgt, _ = full_eth_pair
    runs = []
    for env in ({"ICP_GPU_MATCH_CHUNKS": "1", "ICP_GPU_GROUP_MIN": "0"}, {}, {"ICP_GPU_MATCH_CHUNKS": "3"},
                {"ICP_GPU_MATCH_CHUNKS": "2", "use_graph": 0}, {"ICP_GPU_GROUP_MIN": "1"}, {"ICP_GPU_GROUP_MIN": "32"}):
        for k in ("ICP_GPU_MATCH_CHUNKS", "ICP_GPU_GROUP_MIN"):
            monkeypatch.delenv(k, raising=False)
        for k, v in env.items():
            if k.startswith("ICP_"):
                monkeypatch.setenv(k, v)
        c = capi.Context(0)
        try:
            cfg = capi.default_config()
            cfg.metric, cfg.n_iterations, cfg.max_distance_sq, cfg.nn_algorithm, cfg.collect_stats = 1, 6, 10.0, 2, 0
            cfg.use_graph = env.get("use_graph", 1)
            c.set_config(cfg)
            load(c, src, tgt)
            pose, hist, n_it = c.estimate_pose()
            idx, w = c.query_matches(pose)
            runs.append((pose, hist, idx, w))
        finally:
            c.close()
    for pose, hist, idx, w in runs[1:]:
        assert np.array_equal(pose, runs[0][0]) and np.array_equal(hist, runs[0][1])
        assert np.array_equal(idx, runs[0][2]) and np.array_equal(w, runs[0][3])


def test_reupload_of_the_same_clouds_gives_identical_bits(ctx, full_eth_pair):
    """The index is a function of the cloud alone: the radix sort ranks by (cell code, original index) without atomics, so
    uploading the same pair again (and into a second context) reproduces the correspondences, every pose of the trajectory and
    hence the fp64 summation order bit for bit."""
    src, tgt, _ = full_eth_pair
    cfg = capi.default_config()
    cfg.metric, cfg.n_iterations, cfg.max_distance_sq, cfg.nn_algorithm, cfg.collect_stats = 1, 8, 10.0, 2, 0
    runs = []
    other = capi.Context(0)
    try:
        for c in (ctx, ctx, other):
            c.set_config(cfg)
            load(c, src, tgt)                               # a fresh upload + index build every time
            pose, hist, n_it = c.estimate_pose()
            idx, w = c.query_matches(pose)
            runs.append((pose, hist, idx, w))
    finally:
        other.close()
    for pose, hist, idx, w in runs[1:]:
        assert np.array_equal(pose, runs[0][0]) and np.array_equal(hist, runs[0][1])
        assert np.array_equal(idx, runs[0][2]) and np.array_equal(w, runs[0][3])


def test_config4_full_size_teacher_forced(ctx):
    """configs[3] at FULL size: 370k-point coloured ETH-shaped pair, multi-resolution + symmetric metric + LM + 6-D colour k-NN +
    colour weighting.  The device runs the registration; at five poses of ITS OWN trajectory (first, three in between, last) the
    oracle's stages 2-4 on the level cloud of that iteration must give the same correspondences and weights bit for bit."""
    src, tgt, _ = synth.eth_pair(seed=1234, colors="texture")
    assert len(src) == 370488
    ocfg = orc.Config(metric=2, minimizer=1, weighting=3, color_icp=True, multires=True, max_distance_sq=0.1, n_iterations=6)
    load(ctx, src, tgt)
    cfg = gpu_config(ocfg, nn_algorithm=2)
    ctx.set_config(cfg)
    pose, hist, n_it = ctx.estimate_pose()
    assert n_it >= 6 and np.isfinite(pose).all()
    # the level schedule of ICPOptimizer.h:503-525,634-655: stride halves every iteration until 1
    stride = orc.coarsest_stride(len(src))
    strides = []
    for i in range(n_it):
        strides.append(stride)
        if stride > 1:
            stride = max(stride // 2, 1)
    tree = orc.KdTree(tgt.points, tgt.colors)
    poses = [np.eye(4, dtype=np.float32)] + list(hist)
    flat = capi.default_config()
    for k in sorted({0, n_it // 4, n_it // 2, 3 * n_it // 4, n_it - 1}):
        sel = orc.coarse_indices(src.points, src.normals, strides[k])            # PointCloud::getCoarseResolution (PointCloud.h:325-343)
        om = orc.match_pipeline(ocfg, poses[k], src.points, src.normals, src.colors, tgt.points, tgt.normals, tgt.colors, sel_idx=sel, tree=tree)
        qcfg = gpu_config(ocfg, nn_algorithm=2); qcfg.multires = 0
        ctx.set_config(qcfg)
        idx, w = ctx.query_matches(poses[k], sel_idx=sel)
        assert_matches_equal(idx, w, om, f"iteration {k} (stride {strides[k]}, {len(sel)} points)")
        assert (idx >= 0).sum() > 0.3 * len(sel) or strides[k] > 64
    ctx.set_config(cfg)


def test_point_to_point_centred_data_within_1e_5(ctx, small_eth_pair):
    """Point-to-point against the reference build at the north-star tolerance (1e-5 m): the 3e-5 m this suite allows for that
    metric on 17 m coordinates is the REFERENCE's own fp32 Procrustes noise (means and the 3x3 moment accumulated in fp32,
    t = R(mean_d - mean_s) - R mean_d + mean_d in fp32, ProcrustesAligner.h:13-70) -- with both clouds moved to the origin
    (coordinates within a few metres of 0) it disappears and the fp64-accumulating device agrees within 1e-5.  Where the reference
    build is absent the teacher-forced iterations come from the oracle (oracle/oracle_as_ref.py): the device's point-to-point loop
    against an fp64 restatement, which says nothing about the reference's fp32 noise."""
    from oracle import oracle_as_ref, ref
    R = ref if ref.available() else oracle_as_ref
    src, tgt, _ = small_eth_pair
    c0 = tgt.points[np.isfinite(tgt.points).all(1)].mean(0)
    sp, tp = (src.points - c0).astype(np.float32)[::2], (tgt.points - c0).astype(np.float32)[::2]
    sn, tn = src.normals[::2], tgt.normals[::2]
    z = np.zeros((len(sp), 4), np.uint8); zt = np.zeros((len(tp), 4), np.uint8)
    cfg = capi.default_config()
    cfg.metric, cfg.n_iterations, cfg.max_distance_sq, cfg.nn_algorithm = 0, 4, 0.5, 2
    ctx.set_config(cfg)
    ctx.set_target(tp, tn, zt); ctx.set_source(sp, sn, z)
    pose, hist, n_it = ctx.estimate_pose()
    prev = np.eye(4, dtype=np.float32)
    for k in range(n_it):
        n, pr, _ = R.estimate_pose(0, 0, sp, sn, z, tp, tn, zt, sp[:4], tp[:4], n_iterations=1, max_distance_sq=0.5, init_pose=prev)
        assert n == 1
        assert rot_angle(pr, hist[k]) < 1e-5 and np.abs(pr[:3, 3] - hist[k][:3, 3]).max() < 1e-5, (k, rot_angle(pr, hist[k]), np.abs(pr[:3, 3] - hist[k][:3, 3]).max())
        prev = hist[k]


def test_full_size_tum_projective_bit_exact(ctx):
    """configs[2]: 640x480 frames, projective matching, normals weighting: correspondences bit-exact vs the oracle."""
    src, tgt, k, _ = synth.tum_pair(seed=1234, frame_gap=10)
    assert len(src) == 307200
    ocfg = orc.Config(metric=2, matching=1, weighting=2, max_distance_sq=0.1, n_iterations=1,
                      fx=float(k[0, 0]), fy=float(k[1, 1]), cx=float(k[0, 2]), cy=float(k[1, 2]), width=640, height=480)
    load(ctx, src, tgt)
    ctx.set_camera(k, 640, 480)
    ctx.set_config(gpu_config(ocfg))
    om = orc.match_pipeline(ocfg, np.eye(4, dtype=np.float32), src.points, src.normals, src.colors, tgt.points, tgt.normals, tgt.colors)
    idx, w = ctx.query_matches(np.eye(4, dtype=np.float32))
    assert_matches_equal(idx, w, om)
    assert (om["idx"] > 0).sum() > 100000


def test_config4_multires_symmetric_lm_color(ctx):
    """configs[3]: multi-resolution + symmetric metric + LM + 6-D colour k-NN + colour weighting (reduced size so that
    the oracle's LM with its per-residual jets stays in seconds)."""
    src, tgt, _ = synth.eth_pair(seed=77, n_sweeps=86, n_beams=270, colors="texture")
    ocfg = orc.Config(metric=2, minimizer=1, weighting=3, color_icp=True, multires=True, max_distance_sq=0.1, n_iterations=6)
    rc, opose, ohist, nq = orc.estimate_pose(ocfg, src.points, src.normals, src.colors, tgt.points, tgt.normals, tgt.colors)
    assert rc == 0
    load(ctx, src, tgt)
    ctx.set_config(gpu_config(ocfg, nn_algorithm=2))
    pose, hist, n_it = ctx.estimate_pose()
    assert n_it == len(ohist) and ctx.stats().n_queries == nq
    assert pose_close(pose, opose), f"rot {rot_angle(pose, opose):.2e} trans {np.linalg.norm(pose[:3, 3] - opose[:3, 3]):.2e}"


def test_async_pair_queue_two_contexts(bunny, small_eth_pair):
    """The pair queue of section 8(e): registrations enqueued on two contexts without waiting, fetched later."""
    bs, bt, _, _ = bunny
    es, et, _ = small_eth_pair
    with capi.Context(0) as c1, capi.Context(0) as c2:
        cfg = capi.default_config()
        cfg.metric = 1
        c1.set_config(cfg)
        cfg.max_distance_sq = 0.1
        c2.set_config(cfg)
        c1.set_target(bt.points, bt.normals, bt.colors); c1.set_source(bs.points, bs.normals, bs.colors)
        c2.set_target(et.points, et.normals, et.colors); c2.set_source(es.points, es.normals, es.colors)
        ref1, _, _ = c1.estimate_pose()
        ref2, _, _ = c2.estimate_pose()
        c1.estimate_pose_async(); c2.estimate_pose_async()
        with pytest.raises(capi.IcpGpuError) as e:          # one registration per context at a time
            c1.estimate_pose_async()
        assert e.value.code == capi.E_STATE
        p2, n2 = c2.estimate_pose_finish()
        p1, n1 = c1.estimate_pose_finish()
        assert n1 == 20 and n2 == 20 and np.array_equal(p1, ref1) and np.array_equal(p2, ref2)


# ----------------------------------------------------------------------------- adversarial shapes for the index
def _cloud(kind, n, rng):
    if kind == "uniform":
        return rng.uniform(-1, 1, size=(n, 3)).astype(np.float32)
    if kind == "clustered":      # a few very dense blobs far apart: deep over-full cells, empty space in between
        c = rng.uniform(-50, 50, size=(4, 3))
        return (c[rng.integers(0, 4, n)] + rng.normal(0, 1e-3, size=(n, 3))).astype(np.float32)
    if kind == "identical":      # every point the same: one finest cell holds everything, ties everywhere
        return np.tile(np.array([[0.25, -3.0, 7.5]], np.float32), (n, 1))
    if kind == "line":           # zero extent on two axes
        t = rng.uniform(0, 1, n).astype(np.float32)
        return np.stack([t, np.zeros_like(t), np.full_like(t, 2.0)], 1)
    if kind == "plane_dups":     # quantised plane with many exact duplicates
        p = np.zeros((n, 3), np.float32)
        p[:, :2] = rng.integers(0, 20, size=(n, 2)) * 0.05
        return p
    raise ValueError(kind)


@pytest.mark.parametrize("kind", ["uniform", "clustered", "identical", "line", "plane_dups"])
@pytest.mark.parametrize("n_tgt", [1, 2, 31, 32, 33, 100, 1025, 5000, 40000])
def test_index_edge_shapes_against_brute_force(ctx, kind, n_tgt):
    """The grid / BVH / adjacency construction on degenerate target shapes and sizes, checked against the oracle's literal
    brute-force scan (lowest index on ties), cold and warm-started, with and without a distance threshold."""
    rng = np.random.default_rng(n_tgt * 7 + len(kind))
    tgt = _cloud(kind, n_tgt, rng)
    qry = np.concatenate([_cloud(kind, 300, rng) + rng.normal(0, 0.01, size=(300, 3)).astype(np.float32),
                          rng.uniform(-60, 60, size=(100, 3)).astype(np.float32), tgt[:min(50, n_tgt)]]).astype(np.float32)
    zt, zq = np.zeros_like(tgt), np.zeros_like(qry)
    for max_d2 in (1e30, 0.5):
        ref = orc.knn_brute(tgt, qry, max_d2)
        c = capi.default_config()
        c.nn_algorithm, c.max_distance_sq, c.rejection = 2, max_d2, 0
        ctx.set_config(c)
        ctx.set_target(tgt, zt, None)
        ctx.set_source(qry, zq, None)
        for attempt in range(2):                      # second call is warm-started from the first one's neighbours
            idx, w = ctx.query_matches(np.eye(4, dtype=np.float32))
            assert_matches_equal(idx, w, ref, f"{kind} n={n_tgt} max_d2={max_d2} attempt {attempt}")
        shifted = synth.make_pose([0.01, -0.02, 0.005], [0.3, -0.2, 0.4])      # warm start after a small motion
        q2 = orc.transform_points(shifted, qry)
        ref2 = orc.knn_brute(tgt, q2, max_d2)
        idx, w = ctx.query_matches(shifted)
        assert_matches_equal(idx, w, ref2, f"{kind} n={n_tgt} max_d2={max_d2} shifted")


@pytest.mark.parametrize("group_min", ["1", "8", "0"])
@pytest.mark.parametrize("kind,n_tgt", [("uniform", 5000), ("clustered", 40000), ("plane_dups", 5000), ("line", 1025), ("identical", 100), ("uniform", 33)])
def test_group_search_on_runs_of_far_queries_against_brute_force(kind, n_tgt, group_min, monkeypatch):
    """knn_group_kernel (one shared descent for runs of deferred neighbours, ICP_GPU_GROUP_MIN: 1 = every run, 8 = default, 0 = off)
    on degenerate targets: compact blobs of queries 0.5 - 5 units away from the target (runs of far queries that share their
    candidate leaves), a blob straddling the target, scattered far queries (groups too wide: left to the walk) -- exactly the oracle's
    brute-force answers (lowest index on ties) cold, warm-started and after a small motion, with and without a threshold."""
    monkeypatch.setenv("ICP_GPU_GROUP_MIN", group_min)
    rng = np.random.default_rng(n_tgt * 13 + len(kind) + int(group_min))
    tgt = _cloud(kind, n_tgt, rng)
    centre = tgt.mean(0)
    blobs = [centre + np.array(off, np.float32) + rng.normal(0, s, size=(n, 3)).astype(np.float32)
             for off, s, n in (((0.5, 0.2, 0.1), 0.05, 700), ((3.0, -2.0, 1.0), 0.2, 900), ((0.0, 0.0, 5.0), 0.02, 500), ((0.0, 0.0, 0.0), 0.3, 600))]
    qry = np.concatenate(blobs + [rng.uniform(-60, 60, size=(200, 3)).astype(np.float32), tgt[:min(50, n_tgt)]]).astype(np.float32)
    zt, zq = np.zeros_like(tgt), np.zeros_like(qry)
    c = capi.Context(0)                                   # a fresh context: the knob is read when a search is enqueued
    try:
        for max_d2 in (1e30, 30.0, 2.0):                  # (the group search is launched for thresholds >= 1)
            cfg = capi.default_config()
            cfg.nn_algorithm, cfg.max_distance_sq, cfg.rejection = 2, max_d2, 0
            c.set_config(cfg)
            c.set_target(tgt, zt, None)
            c.set_source(qry, zq, None)
            ref = orc.knn_brute(tgt, qry, max_d2)
            for attempt in range(3):                      # from the second call on warm-started: the fast path defers, the groups form
                idx, w = c.query_matches(np.eye(4, dtype=np.float32))
                assert_matches_equal(idx, w, ref, f"{kind} n={n_tgt} max_d2={max_d2} group_min={group_min} attempt {attempt}")
            for step in (([0.01, -0.02, 0.005], [0.3, -0.2, 0.4]), ([0.05, 0.03, -0.04], [1.0, 0.5, -0.8])):
                moved = synth.make_pose(*step)
                ref2 = orc.knn_brute(tgt, orc.transform_points(moved, qry), max_d2)
                idx, w = c.query_matches(moved)
                assert_matches_equal(idx, w, ref2, f"{kind} n={n_tgt} max_d2={max_d2} group_min={group_min} moved")
    finally:
        c.close()


@pytest.mark.parametrize("minimizer", [0, 1])
def test_early_stop_criterion(ctx, bunny, minimizer):
    """SURVEY.md 8f rank 2: with thresholds set, the loop ends (on the device, inside the replayed graph) after the first iteration whose
    increment is below both; the poses up to there are bit for bit those of the full run, which is unchanged when the thresholds are 0."""
    src, tgt, _, _ = bunny
    load(ctx, src, tgt)
    cfg = capi.default_config()
    cfg.metric, cfg.minimizer, cfg.n_iterations, cfg.max_distance_sq, cfg.nn_algorithm = 1, minimizer, 30, 0.0003, 2
    ctx.set_config(cfg)
    full, hist, n_full = ctx.estimate_pose()
    assert n_full == 30
    steps = [(rot_angle(hist[k], hist[k - 1]), float(np.linalg.norm(hist[k][:3, 3] - hist[k - 1][:3, 3]))) for k in range(1, 30)]
    k_stop = next(k for k, (r, t) in enumerate(steps, start=1) if r < 2e-4 and t < 2e-5)      # an iteration well inside the run
    assert 2 <= k_stop <= 28
    cfg.early_stop_rotation, cfg.early_stop_translation = 1e-3, 1e-4                          # generous: the increment, not the pose difference, is tested
    ctx.set_config(cfg)
    pose, h2, n_it = ctx.estimate_pose()
    assert 1 <= n_it < 30 and len(h2) == n_it
    assert np.array_equal(np.asarray(h2), np.asarray(hist[:n_it])) and np.array_equal(pose, hist[n_it - 1])
    for use_graph in (0, 1):
        cfg.use_graph = use_graph
        ctx.set_config(cfg)
        p3, _, n3 = ctx.estimate_pose()
        assert n3 == n_it and np.array_equal(p3, pose)
