"""GPU tests of batched registration with one configuration per pair (icp_gpu_estimate_pose_batch_configs, csrc/batch.cu):
the reference's whole bunny variant matrix in one call, the Levenberg-Marquardt batch kernel against the oracle, the
multi-resolution schedule and mt19937 selection against the single-pair path, grouping, failure isolation, refusals and the
Python entry points built on it."""
import ctypes as C
import os

import numpy as np
import pytest

from icp_variants_b200 import capi, synth
from icp_variants_b200.optimizer import CeresICPOptimizer
from oracle import oracle as orc

pytestmark = pytest.mark.gpu

TOL = 1e-5     # rad / m
RMSE_TOL = 1e-4
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_outputs.npz")
VARIANTS = [("base", {}), ("random", dict(selection=1, proba=0.5, seed=7, selection_rng=0)), ("distance_weights", dict(weighting=1)),
            ("multires", dict(multires=1))]


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


def config(metric=1, minimizer=0, weighting=0, rejection=1, n_iterations=20, max_d2=0.0003, **kw):
    c = capi.default_config()
    c.metric, c.minimizer, c.weighting, c.rejection, c.n_iterations, c.max_distance_sq = metric, minimizer, weighting, rejection, n_iterations, max_d2
    for k, v in kw.items():
        setattr(c, k, v)
    return c


def subsample(cloud, n, seed=0):
    idx = np.sort(np.random.default_rng(seed).choice(len(cloud.points), n, replace=False))
    return synth.Cloud(cloud.points[idx].copy(), cloud.normals[idx].copy(), None)


def with_nonfinite(cloud):
    """A copy with non-finite points and normals, which the level filter and the mt19937 draw skip."""
    p, n = cloud.points.copy(), cloud.normals.copy()
    p[3::41, 1] = np.nan; p[7::53, 0] = np.inf; n[5::37, 2] = np.nan
    return synth.Cloud(p, n, None)


def raw_batch(ctx, cfgs, ci, sources, targets, rows, poses=None):
    """The C call itself, for arguments the Python wrapper would not build."""
    table = (capi.Config * max(len(cfgs), 1))(*cfgs)
    ci = np.ascontiguousarray(ci, np.int32); B = len(ci)
    sp, sn, so = capi._concat_clouds(sources); tp, tn, to = capi._concat_clouds(targets)
    pin = capi._batch_poses(poses, B); pout = np.zeros((B, 16), np.float32)
    n_it = np.zeros(B, np.int32); st = np.zeros(B, np.int32); hist = np.zeros((B, max(rows, 1), 16), np.float32)
    p = capi._ptr
    return capi.lib().icp_gpu_estimate_pose_batch_configs(ctx._h, len(cfgs), table, B, p(ci), p(sp), p(sn), p(so), p(tp), p(tn), p(to), p(pin),
                                                          p(pout), p(n_it), p(st), p(hist), rows)


def single(ctx, cfg, src, tgt, init):
    ctx.set_config(cfg); ctx.set_source(src.points, src.normals); ctx.set_target(tgt.points, tgt.normals)
    try:
        return ctx.estimate_pose(init)
    except capi.IcpGpuError as e:
        return e.pose, None, e.n_iterations


@pytest.fixture(scope="module")
def ctx():
    with capi.Context(0) as c:
        yield c


@pytest.fixture(scope="module")
def ctx1():
    with capi.Context(0) as c:
        yield c


@pytest.fixture(scope="module")
def golden():
    return np.load(GOLDEN)


def matrix():
    cfgs, keys = [], []
    for mi in (0, 1):
        for me in (0, 1, 2):
            for name, kw in VARIANTS:
                cfgs.append(config(metric=me, minimizer=mi, **kw))
                keys.append(f"bunny_{mi}_{me}_{name}")
    return cfgs, keys


# ------------------------------------------------------------------------------------------------ 1. the matrix in one call
def test_reference_matrix_in_one_call(ctx, bunny, golden):
    src, tgt, gs, gt = bunny
    cfgs, keys = matrix()
    ci = np.tile(np.arange(24, dtype=np.int32), 4)                 # the configurations interleaved, four copies each
    B = len(ci)
    poses, n_it, status, hist = ctx.estimate_pose_batch_configs(cfgs, ci, [src] * B, [tgt] * B, want_history=True)
    assert (status == capi.OK).all() and (n_it == 20).all() and hist.shape == (B, 20, 4, 4)
    ctx.set_correspondences(src.points[gs], tgt.points[gt])
    for b in range(B):
        key = keys[ci[b]]
        assert pose_close(poses[b], golden[key + "_pose"]), (key, rot_angle(poses[b], golden[key + "_pose"]))
        rmse = np.array([ctx.alignment_error(hist[b, i])[0] for i in range(20)])
        assert np.abs(rmse - golden[key + "_rmse"]).max() < RMSE_TOL, key
    for k in range(24):
        copies = np.flatnonzero(ci == k)
        for b in copies[1:]:
            assert np.array_equal(poses[b], poses[copies[0]]) and np.array_equal(hist[b], hist[copies[0]]), keys[k]


# ------------------------------------------------------------------------------------------------ 2. LM against the oracle
def oracle_lm(cfg, src, tgt, init):
    ocfg = orc.Config(metric=cfg.metric, minimizer=1, weighting=cfg.weighting, rejection=cfg.rejection, max_distance_sq=cfg.max_distance_sq,
                      n_iterations=cfg.n_iterations, lm_max_iterations=cfg.lm_max_iterations)
    return orc.estimate_pose(ocfg, src.points, src.normals, src.colors, tgt.points, tgt.normals, tgt.colors, init_pose=init)


LM_CFGS = [config(metric=me, minimizer=1, weighting=w, rejection=r, n_iterations=10) for me in (0, 1, 2) for w in (0, 1, 2) for r in (0, 1)]


def test_lm_free_running_follows_the_oracle(ctx, bunny):
    src, tgt, _, _ = bunny
    starts = [perturbation(100 + s) for s in range(8)]
    ci = np.repeat(np.arange(len(LM_CFGS), dtype=np.int32), len(starts))
    init = np.stack([starts[b % len(starts)] for b in range(len(ci))])
    poses, n_it, status, hist = ctx.estimate_pose_batch_configs(LM_CFGS, ci, [src] * len(ci), [tgt] * len(ci), init, want_history=True)
    for b in range(len(ci)):
        cfg = LM_CFGS[ci[b]]
        rc, opose, ohist, _ = oracle_lm(cfg, src, tgt, init[b])
        what = (cfg.metric, cfg.weighting, cfg.rejection, b % len(starts))
        assert rc == 0 and status[b] == capi.OK and n_it[b] == len(ohist), what
        for k in range(n_it[b]):
            assert pose_close(hist[b, k], ohist[k]), (what, k, rot_angle(hist[b, k], ohist[k]))
        assert np.array_equal(poses[b], hist[b, n_it[b] - 1])


def test_lm_teacher_forced_outer_iteration(ctx, bunny):
    """One outer iteration from every pose of the oracle's trajectory lands on the oracle's next pose."""
    src, tgt, _, _ = bunny
    cfgs, ci, init, want = [], [], [], []
    for k, cfg in enumerate(LM_CFGS):
        rc, _, ohist, _ = oracle_lm(cfg, src, tgt, perturbation(7))
        assert rc == 0
        one = config(metric=cfg.metric, minimizer=1, weighting=cfg.weighting, rejection=cfg.rejection, n_iterations=1)
        cfgs.append(one)
        for i in range(len(ohist) - 1):
            ci.append(k); init.append(ohist[i]); want.append(ohist[i + 1])
    poses, n_it, status = ctx.estimate_pose_batch_configs(cfgs, np.array(ci, np.int32), [src] * len(ci), [tgt] * len(ci), np.stack(init))
    assert (status == capi.OK).all() and (n_it == 1).all()
    for b in range(len(ci)):
        assert pose_close(poses[b], want[b]), (ci[b], rot_angle(poses[b], want[b]))


# ------------------------------------------------------------------------------------------------ 3. batch = single-pair path
SIZES = [150, 250, 450, 900, 1054]          # 1, 2, 3, 4 and 4 pyramid levels


def mixed_pairs(bunny):
    src, tgt, _, _ = bunny
    clouds = [subsample(src, n, seed=n) if n < len(src.points) else src for n in SIZES]
    clouds.append(with_nonfinite(src))
    clouds.append(with_nonfinite(subsample(src, 450, seed=3)))
    return clouds, tgt


SINGLE_CFGS = [
    config(metric=1, minimizer=1, multires=1),
    config(metric=2, minimizer=1, selection=1, proba=0.5, seed=11, selection_rng=0),
    config(metric=0, minimizer=1, multires=1, selection=1, proba=0.6, seed=3, selection_rng=0, n_iterations=6),
    config(metric=0, minimizer=0, multires=1, selection=1, proba=0.5, seed=5, selection_rng=0),
    config(metric=2, minimizer=0, multires=1, n_iterations=8),
    config(metric=1, minimizer=1, multires=1, selection=1, proba=0.7, seed=9, selection_rng=1, n_iterations=5),
]


def test_batch_equals_single_pair_path(ctx, ctx1, bunny):
    clouds, tgt = mixed_pairs(bunny)
    ci = np.array([k for k in range(len(SINGLE_CFGS)) for _ in clouds], np.int32)
    sources = [c for _ in SINGLE_CFGS for c in clouds]
    init = np.stack([perturbation(b) for b in range(len(ci))])
    poses, n_it, status, hist = ctx.estimate_pose_batch_configs(SINGLE_CFGS, ci, sources, [tgt] * len(ci), init, want_history=True)
    for b in range(len(ci)):
        cfg = SINGLE_CFGS[ci[b]]
        pose, shist, sn = single(ctx1, cfg, sources[b], tgt, init[b])
        what = (int(ci[b]), len(sources[b].points), b)
        assert n_it[b] == sn == capi.iterations_bound(cfg, len(sources[b].points)), (what, n_it[b], sn)
        assert status[b] == capi.OK, what
        for k in range(sn):
            assert pose_close(hist[b, k], shist[k]), (what, k, rot_angle(hist[b, k], shist[k]))
        assert pose_close(poses[b], pose), what


# ------------------------------------------------------------------------------------------------ 4. grouping is invisible
def test_grouping_is_invisible(ctx, bunny):
    clouds, tgt = mixed_pairs(bunny)
    cfgs = [config(metric=me, minimizer=mi, multires=mi, n_iterations=6) for mi in (0, 1) for me in (0, 1, 2)]
    ci = np.array([(3 * b + b // 6) % 6 for b in range(18)], np.int32)
    sources = [clouds[b % len(clouds)] for b in range(18)]
    init = np.stack([perturbation(50 + b) for b in range(18)])
    poses, n_it, status, hist = ctx.estimate_pose_batch_configs(cfgs, ci, sources, [tgt] * 18, init, want_history=True)
    for b in range(18):
        p1, n1, s1, h1 = ctx.estimate_pose_batch_configs([cfgs[ci[b]]], np.zeros(1, np.int32), [sources[b]], [tgt], init[b:b + 1], want_history=True)
        assert np.array_equal(poses[b], p1[0]) and n_it[b] == n1[0] and status[b] == s1[0], b
        assert np.array_equal(hist[b, :h1.shape[1]], h1[0]) and not hist[b, h1.shape[1]:].any(), b


# ------------------------------------------------------------------------------------------------ 5. schedule and history
def test_schedule_and_history(ctx, ctx1, bunny):
    clouds, tgt = mixed_pairs(bunny)
    cfgs = [config(metric=1, minimizer=mi, multires=1, n_iterations=2) for mi in (0, 1)]
    ci = np.array([k for k in range(2) for _ in clouds], np.int32)
    sources = [c for _ in cfgs for c in clouds]
    _, n_it, status, hist = ctx.estimate_pose_batch_configs(cfgs, ci, sources, [tgt] * len(ci), want_history=True)
    bounds = [capi.iterations_bound(cfgs[ci[b]], len(sources[b].points)) for b in range(len(ci))]
    assert sorted(set(bounds)) == [2, 3, 4] and hist.shape[1] == 4
    assert (status == capi.OK).all() and n_it.tolist() == bounds
    for b in range(len(ci)):
        assert hist[b, :n_it[b]].any(axis=(1, 2)).all() and not hist[b, n_it[b]:].any()
    for cfg in cfgs + [config(n_iterations=7), config(multires=1, n_iterations=0)]:
        for c in clouds:
            ctx1.set_config(cfg); ctx1.set_source(c.points, c.normals)
            assert capi.iterations_bound(cfg, len(c.points)) == ctx1.max_iterations()
    assert raw_batch(ctx, cfgs, [0, 1], [clouds[3], clouds[3]], [tgt, tgt], 3) == capi.E_ARG    # 4 levels need 4 rows
    assert raw_batch(ctx, cfgs, [0, 1], [clouds[3], clouds[3]], [tgt, tgt], 4) == capi.OK


# ------------------------------------------------------------------------------------------------ 6. failure isolation
def test_failure_isolation(ctx, ctx1, bunny):
    src, tgt, _, _ = bunny
    far = synth.Cloud(tgt.points + np.float32(10.0), tgt.normals, None)      # no match within the threshold
    ctx1.set_config(config(metric=1)); ctx1.set_source(src.points, src.normals); ctx1.set_target(tgt.points, tgt.normals)
    own_before = ctx1.estimate_pose(perturbation(1))
    cfgs = [config(metric=1, minimizer=1, n_iterations=5), config(metric=2, minimizer=0, multires=1, n_iterations=5)]
    init = np.stack([perturbation(b) for b in range(4)])
    poses, n_it, status = ctx1.estimate_pose_batch_configs(cfgs, np.array([0, 0, 1, 0], np.int32), [src] * 4, [tgt, far, tgt, tgt], init)
    assert status.tolist() == [capi.OK, capi.E_NO_MATCHES, capi.OK, capi.OK] and n_it[1] == 0
    assert np.array_equal(poses[1], init[1])
    for b in (0, 2, 3):
        alone = ctx.estimate_pose_batch_configs([cfgs[(0, 0, 1, 0)[b]]], np.zeros(1, np.int32), [src], [tgt], init[b:b + 1])
        assert np.array_equal(poses[b], alone[0][0]) and n_it[b] == alone[1][0]
    own_after = ctx1.estimate_pose(perturbation(1))
    assert np.array_equal(own_before[0], own_after[0]) and np.array_equal(own_before[1], own_after[1])


def test_early_stop_under_lm_and_multires(ctx, ctx1, bunny):
    src, tgt, _, _ = bunny
    cfgs = [config(metric=1, minimizer=1, n_iterations=30, early_stop_rotation=1e-4, early_stop_translation=1e-5),
            config(metric=1, minimizer=0, multires=1, n_iterations=30, early_stop_rotation=1e-4, early_stop_translation=1e-5)]
    init = np.stack([perturbation(3), perturbation(4)])
    poses, n_it, status = ctx.estimate_pose_batch_configs(cfgs, np.array([0, 1], np.int32), [src, src], [tgt, tgt], init)
    assert (status == capi.OK).all() and (n_it < 30).all(), n_it
    for b in range(2):
        pose, _, sn = single(ctx1, cfgs[b], src, tgt, init[b])
        assert sn == n_it[b] and pose_close(poses[b], pose)


# ------------------------------------------------------------------------------------------------ 7. determinism, refusals, forms
def test_two_calls_identical(ctx, bunny):
    clouds, tgt = mixed_pairs(bunny)
    ci = np.arange(len(SINGLE_CFGS), dtype=np.int32).repeat(2)
    sources = [clouds[b % len(clouds)] for b in range(len(ci))]
    a = ctx.estimate_pose_batch_configs(SINGLE_CFGS, ci, sources, [tgt] * len(ci), want_history=True)
    b = ctx.estimate_pose_batch_configs(SINGLE_CFGS, ci, sources, [tgt] * len(ci), want_history=True)
    for x, y in zip(a, b):
        assert np.array_equal(x, y)


def test_refusals(ctx, bunny):
    src, tgt, _, _ = bunny
    ok = config(n_iterations=2)
    for bad in (config(matching=1), config(color_icp=1), config(nn_algorithm=3), config(multires=1, pyramid_mode=1, selection_rng=1),
                config(metric=5), config(lm_max_iterations=65)):
        assert raw_batch(ctx, [ok, bad], [0, 1], [src, src], [tgt, tgt], 20) == capi.E_ARG
        assert "config 1" in capi.lib().icp_gpu_last_error(ctx._h).decode()
    big = synth.Cloud(np.zeros((capi.BATCH_MAX_TARGET + 1, 3), np.float32), None, None)
    assert raw_batch(ctx, [ok], [0, 0], [src, src], [tgt, big], 2) == capi.E_ARG
    assert "pair 1" in capi.lib().icp_gpu_last_error(ctx._h).decode()
    for ci in ([0, 1], [-1, 0]):
        assert raw_batch(ctx, [ok], ci, [src, src], [tgt, tgt], 2) == capi.E_ARG
    assert raw_batch(ctx, [], [0], [src], [tgt], 2) == capi.E_ARG
    assert raw_batch(ctx, [ok], [0], [src], [tgt], 1) == capi.E_ARG                   # history_rows below n_iterations
    # bad offsets
    table = (capi.Config * 1)(ok)
    sp, sn, so = capi._concat_clouds([src, src]); tp, tn, to = capi._concat_clouds([tgt, tgt])
    pin = capi._batch_poses(None, 2); pout = np.zeros((2, 16), np.float32); n = np.zeros(2, np.int32); st = np.zeros(2, np.int32)
    ci = np.zeros(2, np.int32)
    for bad_so in (np.array([1, 1054, 2108], np.int64), np.array([0, 1054, 1000], np.int64)):
        assert capi.lib().icp_gpu_estimate_pose_batch_configs(ctx._h, 1, table, 2, capi._ptr(ci), capi._ptr(sp), capi._ptr(sn), capi._ptr(bad_so),
                                                              capi._ptr(tp), capi._ptr(tn), capi._ptr(to), capi._ptr(pin), capi._ptr(pout),
                                                              capi._ptr(n), capi._ptr(st), None, 0) == capi.E_ARG
    assert capi.lib().icp_gpu_iterations_bound(None, 10) == capi.E_ARG
    assert capi.lib().icp_gpu_iterations_bound(C.byref(ok), -1) == capi.E_ARG


def test_torch_form_equals_host_form(ctx, bunny):
    torch = pytest.importorskip("torch")
    clouds, tgt = mixed_pairs(bunny)
    ci = np.arange(len(SINGLE_CFGS), dtype=np.int32).repeat(2)
    sources = [clouds[b % len(clouds)] for b in range(len(ci))]
    init = np.stack([perturbation(b) for b in range(len(ci))])
    host = ctx.estimate_pose_batch_configs(SINGLE_CFGS, ci, sources, [tgt] * len(ci), init, want_history=True)
    dev = torch.device("cuda", 0)
    sp, sn, so = capi._concat_clouds(sources); tp, tn, to = capi._concat_clouds([tgt] * len(ci))
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)  # noqa: E731
    out = ctx.estimate_pose_batch_configs_dev(SINGLE_CFGS, t(ci), t(sp), t(so), t(tp), t(to), t(sn), t(tn), t(init), want_history=True)
    for x, y in zip(host, out):
        assert np.array_equal(x, y.cpu().numpy())


# ------------------------------------------------------------------------------------------------ 8. Python entry points
def test_ceres_optimizer_batch_equals_estimate_pose(bunny):
    src, tgt, _, _ = bunny
    opt = CeresICPOptimizer(device=0)
    opt.setMetric(2); opt.setNbOfIterations(8); opt.setMatchingMethod(0); opt.setMatchingMaxDistance(0.0003)
    opt.setSelectionMethod(1, 0.5); opt.seed = 13; opt.enableMultiResolution(True)
    init = [perturbation(200 + b) for b in range(4)]
    poses = opt.estimatePoseBatch([src] * 4, [tgt] * 4, np.stack(init))
    assert opt.last_error == [None] * 4
    for b in range(4):
        assert pose_close(poses[b], opt.estimatePose(src, tgt, init[b], calculateRMSE=False)), b


def test_batched_experiment_runner_reproduces_the_reference_matrix(golden, bunny, tmp_path):
    from icp_variants_b200 import experiment as X
    rows = ["expName,expType,useLinear,useMetric,matchingMethod,selectionMethod,weightingMethod,useMultiresolution,numIterations,maxMatchingDist,samplingProba"]
    keys = []
    for lin in (0, 1):
        for metric in (0, 1, 2):
            for name, (sel, wgt, mr, proba) in (("base", (0, 0, 0, 1.0)), ("random", (1, 0, 0, 0.5)), ("distance_weights", (0, 1, 0, 1.0)), ("multires", (0, 0, 1, 1.0))):
                rows.append(f"bunny{len(keys):03d},bunny,{lin},{metric},0,{sel},{wgt},{mr},20,0.0003,{proba}")
                keys.append(f"bunny_{0 if lin else 1}_{metric}_{name}")
    csv = tmp_path / "bunny_experiments.csv"
    csv.write_text("\n".join(rows) + "\n")
    res = X.run_experiments(str(csv), {"bunny": bunny}, out_dir=str(tmp_path), seed=7, batched=True)
    for r, key in zip(res, keys):
        assert pose_close(r["pose"], golden[key + "_pose"]), key
        on_disk = np.loadtxt(r["file"], dtype=np.float32)
        assert len(on_disk) == 20 and np.abs(on_disk - golden[key + "_rmse"]).max() < RMSE_TOL, key
