"""GPU tests of multi-start registration (icp_gpu_estimate_pose_multistart, csrc/multistart.cu): every start against the single-pair
path from the same pose, the scoring pass's matches bit for bit against query_matches and the oracle, independence of the starts
(K, cluster size, failures, early stop), the context's own state, refusals and the Python entry points."""

import numpy as np
import pytest

from icp_variants_b200 import capi, synth
from icp_variants_b200.optimizer import LinearICPOptimizer
from oracle import oracle as orc

pytestmark = pytest.mark.gpu

TOL = 1e-5     # rad / m


def rot_angle(pa, pb):
    d = np.linalg.norm(pa[:3, :3].astype(np.float64) - pb[:3, :3].astype(np.float64))
    return float(2.0 * np.arcsin(min(d / (2.0 * np.sqrt(2.0)), 1.0)))


def pose_close(pa, pb, tol=TOL):
    return rot_angle(pa, pb) <= tol and float(np.abs(pa[:3, 3].astype(np.float64) - pb[:3, 3]).max()) <= tol


def perturbation(seed, max_angle=0.02, max_trans=0.002):
    rng = np.random.default_rng(seed)
    axis = rng.normal(size=3); axis /= np.linalg.norm(axis)
    a = rng.uniform(0.0, max_angle)
    K = np.array([[0, -axis[2], axis[1]], [axis[2], 0, -axis[0]], [-axis[1], axis[0], 0]])
    P = np.eye(4)
    P[:3, :3] = np.eye(3) + np.sin(a) * K + (1 - np.cos(a)) * K @ K
    P[:3, 3] = rng.uniform(-max_trans, max_trans, 3)
    return P.astype(np.float32)


def yaw(deg, t=(0.0, 0.0, 0.0)):
    return synth.make_pose(np.asarray(t, np.float64), (0.0, 0.0, deg)).astype(np.float32)


def config(metric=1, minimizer=0, weighting=0, rejection=1, n_iterations=20, max_d2=0.0003, **kw):
    c = capi.default_config()
    c.metric, c.minimizer, c.weighting, c.rejection, c.n_iterations, c.max_distance_sq = metric, minimizer, weighting, rejection, n_iterations, max_d2
    for k, v in kw.items():
        setattr(c, k, v)
    return c


def bunny_starts():
    """8 seeded perturbations and two far starts."""
    return np.stack([perturbation(s) for s in range(8)] + [perturbation(100, 0.6, 0.05), perturbation(101, 1.2, 0.1)])


def context(src, tgt, cfg, src_rgba=None, tgt_rgba=None):
    ctx = capi.Context(0)
    ctx.set_config(cfg)
    ctx.set_target(tgt.points, tgt.normals, tgt_rgba)
    ctx.set_source(src.points, src.normals, src_rgba)
    return ctx


def single(ctx, pose):
    """estimate_pose from pose: (status, pose, history, n_iterations)."""
    try:
        p, h, n = ctx.estimate_pose(pose, want_history=True)
        return capi.OK, p, h, n
    except capi.IcpGpuError as e:
        return e.code, e.pose, None, e.n_iterations


def check_against_single(ctx, starts):
    res = ctx.estimate_pose_multistart(starts, want_history=True)
    for k, s in enumerate(starts):
        rc, p, h, n = single(ctx, s)
        assert res["status"][k] == rc, (k, res["status"][k], rc)
        assert res["n_iterations"][k] == n, (k, res["n_iterations"][k], n)
        assert pose_close(res["poses"][k], p), (k, rot_angle(res["poses"][k], p))
        if h is not None:
            for i in range(n):
                assert pose_close(res["history"][k, i], h[i]), (k, i)
        assert not res["history"][k, n:].any()
    return res


@pytest.mark.parametrize("minimizer", [0, 1])
@pytest.mark.parametrize("metric", [0, 1, 2])
def test_each_start_equals_the_single_path(bunny, minimizer, metric):
    src, tgt, _, _ = bunny
    ctx = context(src, tgt, config(metric=metric, minimizer=minimizer))
    check_against_single(ctx, bunny_starts())


@pytest.mark.parametrize("variant", ["mt19937", "device_stream", "stride_pyramid", "voxel_pyramid", "lm_multires_mt"])
def test_selection_and_pyramids_equal_the_single_path(bunny, variant):
    src, tgt, _, _ = bunny
    kw = {"mt19937": dict(selection=1, proba=0.5, seed=7, selection_rng=0),
          "device_stream": dict(selection=1, proba=0.5, seed=7, selection_rng=1),
          "stride_pyramid": dict(multires=1),
          "voxel_pyramid": dict(multires=1, pyramid_mode=1),
          "lm_multires_mt": dict(minimizer=1, multires=1, selection=1, proba=0.7, seed=3, selection_rng=0)}[variant]
    ctx = context(src, tgt, config(**kw))
    check_against_single(ctx, bunny_starts()[:6])


def check_matches(ctx, res, src_pts, tgt_pts, src_rgba=None, tgt_rgba=None):
    """match_idx / match_w against query_matches bit for bit; inliers and rmse against numpy over those matches."""
    for k, pose in enumerate(res["poses"]):
        idx, w = ctx.query_matches(pose)
        assert np.array_equal(res["match_idx"][k], idx), k
        assert np.array_equal(res["match_w"][k].view(np.int32), w.view(np.int32)), k
        keep = idx >= 0
        assert res["inliers"][k] == int(keep.sum()), k
        if not keep.any():
            assert np.isnan(res["rmse"][k])
            continue
        P = pose.astype(np.float32)
        s = src_pts[keep].astype(np.float32)
        x = ((P[0, 0] * s[:, 0] + P[0, 1] * s[:, 1]) + P[0, 2] * s[:, 2]) + P[0, 3]
        y = ((P[1, 0] * s[:, 0] + P[1, 1] * s[:, 1]) + P[1, 2] * s[:, 2]) + P[1, 3]
        z = ((P[2, 0] * s[:, 0] + P[2, 1] * s[:, 1]) + P[2, 2] * s[:, 2]) + P[2, 3]
        t = tgt_pts[idx[keep]].astype(np.float32)
        dx, dy, dz = x - t[:, 0], y - t[:, 1], z - t[:, 2]
        d2 = (dx * dx + dy * dy) + dz * dz
        if src_rgba is not None:
            for c in range(3):
                e = np.float32(1.0 / 255.0) * src_rgba[keep, c].astype(np.float32) - np.float32(1.0 / 255.0) * tgt_rgba[idx[keep], c].astype(np.float32)
                d2 = d2 + e * e
        want = np.sqrt(np.mean(d2.astype(np.float64)))
        assert abs(res["rmse"][k] - want) <= 1e-12 * want, (k, res["rmse"][k], want)


def test_matches_bit_exact_bunny(bunny):
    src, tgt, _, _ = bunny
    ctx = context(src, tgt, config(weighting=1))
    res = ctx.estimate_pose_multistart(bunny_starts(), want_matches=True)
    check_matches(ctx, res, src.points, tgt.points)


@pytest.mark.parametrize("colour", [False, True])
@pytest.mark.parametrize("max_d2", [0.1, 10.0])
def test_matches_bit_exact_eth(small_eth_pair, colour, max_d2):
    src, tgt, _ = small_eth_pair
    sc = synth.procedural_colors(src.points, seed=5) if colour else None
    tc = synth.procedural_colors(tgt.points, seed=6) if colour else None
    ctx = context(src, tgt, config(metric=1, max_d2=max_d2, color_icp=int(colour), weighting=3 if colour else 0, n_iterations=10),
                  src_rgba=sc, tgt_rgba=tc)
    starts = np.stack([yaw(a, (0.05 * i, 0.0, 0.0)) for i, a in enumerate((-6.0, -2.0, 0.0, 3.0, 8.0))])
    res = ctx.estimate_pose_multistart(starts, want_matches=True)
    check_matches(ctx, res, src.points, tgt.points, sc, tc)


def test_matches_bit_exact_ties_duplicates_nonfinite():
    rng = np.random.default_rng(11)
    t = np.round(rng.uniform(-1, 1, (6000, 3)) * 8.0) / 8.0            # a quantised target: equal distances everywhere
    t = np.concatenate([t, t[:500]]).astype(np.float32)                  # duplicates
    t[7::97, 0] = np.nan; t[11::89, 2] = np.inf
    s = (np.round(rng.uniform(-1, 1, (3000, 3)) * 16.0) / 16.0).astype(np.float32)
    s[5::61, 1] = np.nan
    tgt = synth.Cloud(t, np.tile(np.float32([0, 0, 1]), (len(t), 1)), None)
    src = synth.Cloud(s, np.tile(np.float32([0, 0, 1]), (len(s), 1)), None)
    ctx = context(src, tgt, config(metric=0, rejection=0, max_d2=0.05, n_iterations=3, nn_algorithm=2))
    res = ctx.estimate_pose_multistart(np.stack([np.eye(4, dtype=np.float32), yaw(1.0), yaw(-3.0, (0.01, 0, 0))]), want_matches=True)
    check_matches(ctx, res, src.points, tgt.points)


def test_matches_bit_exact_full_eth_pair_24_yaw_starts():
    src, tgt, _ = synth.eth_pair(seed=1234)
    sub = synth.Cloud(src.points[::32].copy(), src.normals[::32].copy(), None)
    ctx = context(sub, tgt, config(metric=1, max_d2=10.0, n_iterations=30))
    starts = np.stack([yaw(a) for a in np.linspace(-30.0, 30.0, 24)])
    res = ctx.estimate_pose_multistart(starts, want_matches=True)
    check_matches(ctx, res, sub.points, tgt.points)
    rc, p, _, n = single(ctx, starts[3])
    assert rc == res["status"][3] and n == res["n_iterations"][3] and pose_close(res["poses"][3], p)


def test_teacher_forced_against_the_oracle(bunny):
    src, tgt, _, _ = bunny
    ocfg = orc.Config(metric=1, max_distance_sq=0.0003, n_iterations=20)
    rc, _, hist, _ = orc.estimate_pose(ocfg, src.points, src.normals, src.colors, tgt.points, tgt.normals, tgt.colors, init_pose=perturbation(3))
    assert rc == 0
    poses = np.concatenate([perturbation(3)[None], hist]).astype(np.float32)
    ctx = context(src, tgt, config(metric=1, n_iterations=0))
    res = ctx.estimate_pose_multistart(poses, want_matches=True)
    assert (res["n_iterations"] == 0).all() and np.array_equal(res["poses"], poses)
    for k, pose in enumerate(poses):
        om = orc.match_pipeline(ocfg, pose, src.points, src.normals, src.colors, tgt.points, tgt.normals, tgt.colors)
        assert np.array_equal(res["match_idx"][k], om["idx"]), k
        assert np.array_equal(res["match_w"][k].view(np.int32), om["weight"].view(np.int32)), k


def test_a_start_is_the_same_bits_alone_among_many_and_again(bunny):
    src, tgt, _, _ = bunny
    ctx = context(src, tgt, config(metric=2, minimizer=0))
    probe = perturbation(42)
    others = [perturbation(1000 + i, 0.1, 0.01) for i in range(300)]

    def run(K):
        starts = np.stack([probe] + others[:K - 1])
        r = ctx.estimate_pose_multistart(starts, want_history=True, want_matches=True)
        return [r[f][0].tobytes() for f in ("poses", "n_iterations", "status", "inliers", "rmse", "history", "match_idx", "match_w")]

    alone = run(1)
    assert run(16) == alone
    assert run(300) == alone
    assert run(1) == alone


def test_a_failed_start_leaves_its_neighbours_alone(bunny):
    src, tgt, _, _ = bunny
    ctx = context(src, tgt, config())
    far = np.eye(4, dtype=np.float32); far[:3, 3] = 100.0
    starts = np.stack([perturbation(1), far, perturbation(2)])
    res = ctx.estimate_pose_multistart(starts)
    assert list(res["status"]) == [capi.OK, capi.E_NO_MATCHES, capi.OK]
    assert res["n_iterations"][1] == 0 and np.array_equal(res["poses"][1], far) and res["inliers"][1] == 0
    ref = ctx.estimate_pose_multistart(starts[[0, 2]])
    assert np.array_equal(ref["poses"], res["poses"][[0, 2]])
    assert res["best"] in (0, 2)


def test_early_stop_per_start(bunny):
    src, tgt, _, _ = bunny
    ctx = context(src, tgt, config(n_iterations=60, early_stop_rotation=1e-4, early_stop_translation=1e-5))
    res = check_against_single(ctx, np.stack([perturbation(1), perturbation(100, 0.3, 0.03), perturbation(5)]))
    assert (res["n_iterations"] < 60).any()


def test_the_context_is_left_alone(bunny):
    src, tgt, _, _ = bunny
    ctx = context(src, tgt, config(metric=1))
    before = ctx.estimate_pose(perturbation(9))
    ctx.estimate_pose_multistart(bunny_starts())
    after = ctx.estimate_pose(perturbation(9))
    assert before[0].tobytes() == after[0].tobytes() and before[1].tobytes() == after[1].tobytes()
    ctx.estimate_pose_async(perturbation(9))
    with pytest.raises(capi.IcpGpuError) as e:
        ctx.estimate_pose_multistart(bunny_starts())
    assert e.value.code == capi.E_STATE and "pending" in str(e.value)
    ctx.estimate_pose_finish()


def raw(ctx, K, **override):
    n = max(ctx.n_source, 1)
    a = dict(pin=np.tile(np.eye(4, dtype=np.float32).reshape(16), (max(K, 1), 1)), pout=np.zeros((max(K, 1), 16), np.float32),
             n_it=np.zeros(max(K, 1), np.int32), status=np.zeros(max(K, 1), np.int32), inl=np.zeros(max(K, 1), np.int64),
             rmse=np.zeros(max(K, 1)), hist=None, idx=None, w=None)
    a.update(override)
    p = capi._ptr
    return capi.lib().icp_gpu_estimate_pose_multistart(ctx._h, K, p(a["pin"]), p(a["pout"]), p(a["n_it"]), p(a["status"]), p(a["inl"]),
                                                       p(a["rmse"]), p(a["hist"]), p(a["idx"]), p(a["w"])), capi.lib().icp_gpu_last_error(ctx._h).decode()


def test_refusals_and_edge_cases(bunny):
    src, tgt, _, _ = bunny
    ctx = capi.Context(0)
    ctx.set_config(config())
    rc, msg = raw(ctx, 2)
    assert rc == capi.E_STATE and "source" in msg
    ctx.set_source(src.points, src.normals)
    rc, msg = raw(ctx, 2)
    assert rc == capi.E_STATE and "target" in msg
    ctx.set_target(tgt.points, tgt.normals)
    assert raw(ctx, 0)[0] == capi.OK
    rc, msg = raw(ctx, -1)
    assert rc == capi.E_ARG and "n_starts" in msg
    rc, msg = raw(ctx, 2, pout=None)
    assert rc == capi.E_ARG and "required" in msg
    rc, msg = raw(ctx, 2, idx=np.zeros((2, len(src.points)), np.int32))
    assert rc == capi.E_ARG and "together" in msg
    ctx.set_config(config(matching=1))
    rc, msg = raw(ctx, 2)
    assert rc == capi.E_ARG and "projective" in msg
    ctx.set_config(config(nn_algorithm=3))
    rc, msg = raw(ctx, 2)
    assert rc == capi.E_ARG and "norm" in msg
    ctx.set_config(config())
    big = 0x7fffffff // len(src.points) + 1
    rc, msg = raw(ctx, big, pin=np.zeros((1, 16), np.float32))
    assert rc == capi.E_ARG and "INT32_MAX" in msg
    assert capi.lib().icp_gpu_estimate_pose_multistart(None, 1, None, None, None, None, None, None, None, None, None) == capi.E_ARG


def test_attached_peers_are_refused(bunny):
    src, tgt, _, _ = bunny
    ctx = context(src, tgt, config())
    try:
        ctx.peer_attach_ptrs(0, 2, [ctx.peer_address(), ctx.peer_address()])
    except capi.IcpGpuError as e:
        pytest.skip(f"one context cannot stand for two ranks here: {e}")
    try:
        rc, msg = raw(ctx, 1)
        assert rc == capi.E_ARG and "peers" in msg
    finally:
        ctx.peer_detach()


def test_empty_source_behaves_like_estimate_pose(bunny):
    _, tgt, _, _ = bunny
    ctx = capi.Context(0)
    ctx.set_config(config())
    ctx.set_target(tgt.points, tgt.normals)
    ctx.set_source(np.zeros((0, 3), np.float32))
    rc, p, _, n = single(ctx, perturbation(1))
    res = ctx.estimate_pose_multistart(np.stack([perturbation(1)]))
    assert res["status"][0] == rc and res["n_iterations"][0] == n and np.array_equal(res["poses"][0], p)
    assert res["inliers"][0] == 0 and np.isnan(res["rmse"][0])


def test_scorer_and_best(bunny):
    src, tgt, _, _ = bunny
    ctx = context(src, tgt, config(n_iterations=0))
    starts = np.stack([perturbation(100, 0.6, 0.05), np.eye(4, dtype=np.float32), perturbation(101, 1.2, 0.1)])
    res = ctx.estimate_pose_multistart(starts)
    assert res["best"] == int(np.lexsort((np.arange(3), np.nan_to_num(res["rmse"], nan=np.inf), -res["inliers"]))[0])
    assert capi.best_start([5, 5, 7], [0.1, 0.2, np.nan]) == 2 and capi.best_start([5, 5], [0.2, 0.1]) == 1
    assert capi.best_start([], []) == -1


def test_dev_form_and_optimizer(bunny):
    import torch
    src, tgt, _, _ = bunny
    ctx = context(src, tgt, config(metric=1))
    starts = bunny_starts()
    host = ctx.estimate_pose_multistart(starts, want_history=True, want_matches=True)
    dev = ctx.estimate_pose_multistart_dev(torch.from_numpy(starts).cuda(), want_history=True, want_matches=True)
    for f in ("poses", "n_iterations", "status", "inliers", "rmse", "history", "match_idx", "match_w"):
        assert np.array_equal(dev[f].cpu().numpy(), host[f], equal_nan=f == "rmse"), f
    assert dev["best"] == host["best"]
    opt = LinearICPOptimizer(device=0)
    opt.setMetric(1); opt.setNbOfIterations(20); opt.setMatchingMaxDistance(0.0003)
    pose, best, res = opt.estimatePoseMultiStart(src, tgt, starts)
    want = context(src, tgt, opt.config()).estimate_pose_multistart(starts)
    assert best == want["best"] and np.array_equal(pose, want["poses"][best]) and np.array_equal(res["inliers"], want["inliers"])
