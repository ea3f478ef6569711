"""GPU tests of indexed batched registration (icp_gpu_estimate_pose_batch_indexed, csrc/batch_indexed_api.cu and the batch variant of
csrc/multistart.cu): every pair bit for bit against estimate_pose_multistart with one start on a context holding that pair, on batches
that mix bunny pairs with ETH-shaped pairs above the 8192-point limit of estimate_pose_batch; the matches against query_matches and the
oracle; independence of a pair from its neighbours and the order; edge cases, the context's own state, refusals and the other forms."""

import numpy as np
import pytest

from icp_variants_b200 import capi, synth
from icp_variants_b200.optimizer import LinearICPOptimizer
from oracle import oracle as orc

pytestmark = pytest.mark.gpu


def perturbation(seed, max_angle=0.02, max_trans=0.002):
    rng = np.random.default_rng(seed)
    axis = rng.normal(size=3); axis /= np.linalg.norm(axis)
    a = rng.uniform(0.0, max_angle)
    K = np.array([[0, -axis[2], axis[1]], [axis[2], 0, -axis[0]], [-axis[1], axis[0], 0]])
    P = np.eye(4)
    P[:3, :3] = np.eye(3) + np.sin(a) * K + (1 - np.cos(a)) * K @ K
    P[:3, 3] = rng.uniform(-max_trans, max_trans, 3)
    return P.astype(np.float32)


def config(metric=1, minimizer=0, weighting=0, rejection=1, n_iterations=12, max_d2=0.003, **kw):
    c = capi.default_config()
    c.metric, c.minimizer, c.weighting, c.rejection, c.n_iterations, c.max_distance_sq = metric, minimizer, weighting, rejection, n_iterations, max_d2
    for k, v in kw.items():
        setattr(c, k, v)
    return c


@pytest.fixture(scope="module")
def mixed(bunny):
    """Two bunny pairs and three ETH-shaped pairs of ~12.9k points (targets above 8192), with colours, and one start each."""
    src, tgt, _, _ = bunny
    sources, targets, poses = [], [], []
    for i in range(2):
        sources.append(synth.Cloud(src.points, src.normals, synth.procedural_colors(src.points, seed=10 + i)))
        targets.append(synth.Cloud(tgt.points, tgt.normals, synth.procedural_colors(tgt.points, seed=20 + i)))
        poses.append(perturbation(i))
    for seed in (3, 4, 5):
        s, t, _ = synth.eth_pair(seed=seed, n_sweeps=12, n_beams=1077, colors=True)
        assert len(t) > capi.BATCH_MAX_TARGET
        sources.append(s); targets.append(t); poses.append(perturbation(50 + seed, 0.01, 0.02))
    return sources, targets, np.stack(poses)


def reference(cfg, src, tgt, pose):
    """estimate_pose_multistart with K = 1 on a context holding the pair."""
    with capi.Context(0) as ctx:
        ctx.set_config(cfg)
        ctx.set_target(tgt.points, tgt.normals, getattr(tgt, "colors", None))
        ctx.set_source(src.points, src.normals, getattr(src, "colors", None))
        return ctx.estimate_pose_multistart(pose[None], want_history=True, want_matches=True)


def bits(x):
    x = np.ascontiguousarray(x)
    return x.view({4: np.int32, 8: np.int64}[x.dtype.itemsize])


def assert_pair_equal(res, b, ref):
    assert np.array_equal(bits(res["poses"][b]), bits(ref["poses"][0])), b
    assert res["n_iterations"][b] == ref["n_iterations"][0], b
    assert res["status"][b] == ref["status"][0], b
    assert res["inliers"][b] == ref["inliers"][0], b
    assert bits(res["rmse"][b:b + 1])[0] == bits(ref["rmse"][:1])[0], (b, res["rmse"][b], ref["rmse"][0])
    r = ref["history"].shape[1]
    if "history" in res:
        assert np.array_equal(bits(res["history"][b, :r]), bits(ref["history"][0])), b
        assert not res["history"][b, r:].any(), b
    if "match_idx" in res:
        assert np.array_equal(res["match_idx"][b], ref["match_idx"][0]), b
        assert np.array_equal(bits(res["match_w"][b]), bits(ref["match_w"][0])), b


def check_batch(cfg, sources, targets, poses):
    with capi.Context(0) as ctx:
        ctx.set_config(cfg)
        res = ctx.estimate_pose_batch_indexed(sources, targets, poses, want_history=True, want_matches=True)
    for b in range(len(sources)):
        assert_pair_equal(res, b, reference(cfg, sources[b], targets[b], poses[b]))
    return res


@pytest.mark.parametrize("minimizer", [0, 1])
@pytest.mark.parametrize("metric", [0, 1, 2])
def test_each_pair_equals_multistart(mixed, minimizer, metric):
    check_batch(config(metric=metric, minimizer=minimizer), *mixed)


@pytest.mark.parametrize("variant", ["mt19937", "device_stream", "stride_pyramid", "voxel_pyramid", "lm_multires_mt", "colour",
                                     "weighting", "no_rejection", "early_stop"])
def test_selection_pyramids_and_options_equal_multistart(mixed, variant):
    kw = {"mt19937": dict(selection=1, proba=0.5, seed=7, selection_rng=0),
          "device_stream": dict(selection=1, proba=0.5, seed=7, selection_rng=1),
          "stride_pyramid": dict(multires=1),
          "voxel_pyramid": dict(multires=1, pyramid_mode=1),
          "lm_multires_mt": dict(minimizer=1, multires=1, selection=1, proba=0.7, seed=3, selection_rng=0),
          "colour": dict(color_icp=1, weighting=3),
          "weighting": dict(weighting=1),
          "no_rejection": dict(rejection=0),
          "early_stop": dict(early_stop_rotation=1e-4, early_stop_translation=1e-5, n_iterations=30)}[variant]
    res = check_batch(config(**kw), *mixed)
    if variant == "early_stop":
        assert (res["n_iterations"] < 30).any()


@pytest.mark.parametrize("weighting", [2, 3])
def test_other_weightings_equal_multistart(mixed, weighting):
    sources, targets, poses = mixed
    check_batch(config(weighting=weighting, color_icp=1 if weighting == 3 else 0), sources[1:4], targets[1:4], poses[1:4])


def ties_pair():
    rng = np.random.default_rng(11)
    t = np.round(rng.uniform(-1, 1, (6000, 3)) * 8.0) / 8.0            # a quantised target: equal distances everywhere
    t = np.concatenate([t, t[:500]]).astype(np.float32)                  # duplicates
    t[7::97, 0] = np.nan; t[11::89, 2] = np.inf
    s = (np.round(rng.uniform(-1, 1, (3000, 3)) * 16.0) / 16.0).astype(np.float32)
    s[5::61, 1] = np.nan
    z = np.float32([0, 0, 1])
    return synth.Cloud(s, np.tile(z, (len(s), 1)), None), synth.Cloud(t, np.tile(z, (len(t), 1)), None)


def test_matches_equal_query_matches_and_the_oracle(bunny):
    src, tgt, _, _ = bunny
    ts, tt = ties_pair()
    cfg = config(metric=0, rejection=0, max_d2=0.05, n_iterations=0, nn_algorithm=2)
    sources, targets = [ts, src, ts], [tt, tgt, tt]
    poses = np.stack([np.eye(4, dtype=np.float32), perturbation(3), perturbation(4, 0.05, 0.01)])
    with capi.Context(0) as ctx:
        ctx.set_config(cfg)
        res = ctx.estimate_pose_batch_indexed(sources, targets, poses, want_matches=True)
    assert (res["n_iterations"] == 0).all() and np.array_equal(res["poses"], poses)
    ocfg = orc.Config(metric=0, rejection=0, max_distance_sq=0.05, n_iterations=0)
    for b, (s, t) in enumerate(zip(sources, targets)):
        with capi.Context(0) as ctx:
            ctx.set_config(cfg)
            ctx.set_target(t.points, t.normals); ctx.set_source(s.points, s.normals)
            idx, w = ctx.query_matches(poses[b])
        assert np.array_equal(res["match_idx"][b], idx), b
        assert np.array_equal(bits(res["match_w"][b]), bits(w)), b
        assert res["inliers"][b] == int((idx >= 0).sum()), b
        om = orc.match_pipeline(ocfg, poses[b], s.points, s.normals, None, t.points, t.normals, None)
        assert np.array_equal(res["match_idx"][b], om["idx"]), b


def test_a_pair_is_the_same_bits_alone_among_many_in_another_order_and_beside_a_failure(mixed):
    sources, targets, poses = mixed
    cfg = config(metric=2)
    empty = synth.Cloud(np.zeros((0, 3), np.float32), np.zeros((0, 3), np.float32), None)
    with capi.Context(0) as ctx:
        ctx.set_config(cfg)
        alone = ctx.estimate_pose_batch_indexed(sources[3:4], targets[3:4], poses[3:4], want_history=True, want_matches=True)
        many = ctx.estimate_pose_batch_indexed(sources * 6, targets * 6, np.concatenate([poses] * 6), want_history=True, want_matches=True)
        perm = [4, 2, 0, 3, 1]
        shuffled = ctx.estimate_pose_batch_indexed([sources[i] for i in perm] + [sources[0]], [targets[i] for i in perm] + [empty],
                                                   np.concatenate([poses[perm], poses[:1]]), want_history=True, want_matches=True)
    for b in (3, 3 + 5, 3 + 5 * 5):
        assert_pair_equal(many, b, alone)
    assert_pair_equal(shuffled, perm.index(3), alone)
    assert shuffled["status"][5] == capi.E_NO_MATCHES and shuffled["inliers"][5] == 0 and np.isnan(shuffled["rmse"][5])


def test_edge_cases(bunny):
    src, tgt, _, _ = bunny
    cfg = config()
    empty = synth.Cloud(np.zeros((0, 3), np.float32), np.zeros((0, 3), np.float32), None)
    with capi.Context(0) as ctx:
        ctx.set_config(cfg)
        r0 = ctx.estimate_pose_batch_indexed([], [], None, want_history=True, want_matches=True)
        assert len(r0["poses"]) == 0 and r0["best"] == -1
        res = ctx.estimate_pose_batch_indexed([empty, src, src], [tgt, empty, tgt], np.stack([np.eye(4, dtype=np.float32)] * 3), want_history=True,
                                              want_matches=True)
    for b, (s, t) in enumerate([(empty, tgt), (src, empty)]):
        assert_pair_equal(res, b, reference(cfg, s, t, np.eye(4, dtype=np.float32)))
    assert res["status"][2] == capi.OK and res["best"] == 2


def test_the_context_is_left_as_it_was(bunny, mixed):
    src, tgt, _, _ = bunny
    cfg = config()
    with capi.Context(0) as ctx:
        ctx.set_config(cfg)
        ctx.set_target(tgt.points, tgt.normals); ctx.set_source(src.points, src.normals)
        before = ctx.estimate_pose(perturbation(9), want_history=True)
        ctx.estimate_pose_batch_indexed(*mixed)
        after = ctx.estimate_pose(perturbation(9), want_history=True)
        assert np.array_equal(bits(before[0]), bits(after[0])) and before[2] == after[2]
        assert np.array_equal(bits(before[1]), bits(after[1]))


def test_refusals(bunny):
    src, tgt, _, _ = bunny
    L = capi.lib()
    sp = np.ascontiguousarray(src.points, np.float32); tp = np.ascontiguousarray(tgt.points, np.float32)
    so = np.array([0, len(sp)], np.int64); to = np.array([0, len(tp)], np.int64)
    pin = np.eye(4, dtype=np.float32).reshape(1, 16).copy()
    pout = np.zeros((1, 16), np.float32); n_it = np.zeros(1, np.int32); st = np.zeros(1, np.int32)
    inl = np.zeros(1, np.int64); rmse = np.zeros(1, np.float64); hist = np.zeros((1, 40, 16), np.float32)
    midx = np.zeros(len(sp), np.int32); mw = np.zeros(len(sp), np.float32)
    p = capi._ptr

    def call(ctx, B=1, so=so, to=to, sx=sp, tx=tp, pin=pin, inl=inl, hist=None, rows=0, midx=None, mw=None):
        rc = L.icp_gpu_estimate_pose_batch_indexed(ctx._h, B, p(sx), None, None, p(so), p(tx), None, None, p(to), p(pin), p(pout), p(n_it), p(st),
                                                   p(inl), p(rmse), p(hist), rows, p(midx), p(mw))
        return rc, L.icp_gpu_last_error(ctx._h).decode()

    with capi.Context(0) as ctx:
        ctx.set_config(config())
        cases = [(dict(B=-1), "n_pairs -1"),
                 (dict(inl=None), "are required"),
                 (dict(sx=None), "null point array"),
                 (dict(tx=None), "null point array"),
                 (dict(midx=midx), "go together"),
                 (dict(so=np.array([1, len(sp)], np.int64)), "must start at 0"),
                 (dict(B=2, so=np.array([0, 10, 5], np.int64), to=np.array([0, 5, 10], np.int64),
                       pin=np.tile(pin, (2, 1)), inl=np.zeros(2, np.int64)), "not monotone"),
                 (dict(hist=hist, rows=3), "history_rows 3")]
        for kw, msg in cases:
            rc, err = call(ctx, **kw)
            assert rc == capi.E_ARG and msg in err, (kw.keys(), rc, err)
        for field, value, msg in (("matching", 1, "k-NN matching only"), ("nn_algorithm", 3, "squared-distance matching only")):
            c = config(); setattr(c, field, value)
            ctx.set_config(c)
            rc, err = call(ctx)
            assert rc == capi.E_ARG and msg in err, (field, rc, err)
        ctx.set_config(config())
        assert call(ctx, B=0)[0] == capi.OK
        ctx.set_target(tgt.points, tgt.normals); ctx.set_source(src.points, src.normals)
        ctx.estimate_pose_async(np.eye(4, dtype=np.float32))
        rc, err = call(ctx)
        assert rc == capi.E_STATE and "pending" in err
        ctx.estimate_pose_finish()
        assert call(ctx, hist=hist, rows=40, midx=midx, mw=mw)[0] == capi.OK
        # attached peers: one context's mailbox standing for both ranks of a world of two
        try:
            ctx.peer_attach_ptrs(0, 2, [ctx.peer_address(), ctx.peer_address()])
        except capi.IcpGpuError as e:
            pytest.skip(f"one context cannot stand for two ranks here: {e}")
        try:
            rc, err = call(ctx)
            assert rc == capi.E_ARG and "attached peers" in err, (rc, err)
        finally:
            ctx.peer_detach()


def test_size_refusals_before_any_upload():
    L = capi.lib()
    with capi.Context(0) as ctx:
        ctx.set_config(config())
        big = np.array([0, 0x7fffffff // 4 + 1], np.int64)
        z = np.array([0, 0], np.int64)
        pin = np.eye(4, dtype=np.float32).reshape(1, 16).copy()
        o = [np.zeros(16, np.float32), np.zeros(1, np.int32), np.zeros(1, np.int32), np.zeros(1, np.int64), np.zeros(1, np.float64)]
        dummy = np.zeros(3, np.float32)
        p = capi._ptr
        rc = L.icp_gpu_estimate_pose_batch_indexed(ctx._h, 1, p(dummy), None, None, p(z), p(dummy), None, None, p(big), p(pin), *[p(x) for x in o],
                                                   None, 0, None, None)
        assert rc == capi.E_ARG and "above a cloud's limit" in L.icp_gpu_last_error(ctx._h).decode()
        many = np.arange(0, 6 * (0x7fffffff // 4) + 1, 0x7fffffff // 4, dtype=np.int64)      # 6 pairs at the limit: above INT32_MAX in all
        zz = np.zeros(len(many), np.int64)
        pin6 = np.tile(pin, (6, 1)); o6 = [np.zeros((6, 16), np.float32), np.zeros(6, np.int32), np.zeros(6, np.int32), np.zeros(6, np.int64),
                                           np.zeros(6, np.float64)]
        rc = L.icp_gpu_estimate_pose_batch_indexed(ctx._h, 6, p(dummy), None, None, p(many), p(dummy), None, None, p(zz), p(pin6), *[p(x) for x in o6],
                                                   None, 0, None, None)
        assert rc == capi.E_ARG and "exceed INT32_MAX" in L.icp_gpu_last_error(ctx._h).decode()


def test_dev_form_equals_the_host_form_and_the_optimizer_method(mixed):
    import torch
    sources, targets, poses = mixed
    cfg = config(metric=2, multires=1, selection=1, proba=0.6, seed=5, selection_rng=0)
    with capi.Context(0) as ctx:
        ctx.set_config(cfg)
        host = ctx.estimate_pose_batch_indexed(sources, targets, poses, want_history=True, want_matches=True)
        dev = torch.device("cuda", 0)

        def cat(clouds, attr, dtype):
            return torch.from_numpy(np.concatenate([getattr(c, attr) for c in clouds]).astype(dtype)).to(dev)

        off = lambda clouds: torch.tensor(np.concatenate([[0], np.cumsum([len(c) for c in clouds])]), dtype=torch.int64, device=dev)
        d = ctx.estimate_pose_batch_indexed_dev(cat(sources, "points", np.float32), off(sources), cat(targets, "points", np.float32), off(targets),
                                                cat(sources, "normals", np.float32), cat(targets, "normals", np.float32),
                                                cat(sources, "colors", np.uint8), cat(targets, "colors", np.uint8),
                                                torch.from_numpy(poses).to(dev), want_history=True, want_matches=True)
    for k in ("poses", "n_iterations", "status", "inliers", "rmse", "history"):
        assert np.array_equal(bits(d[k].cpu().numpy()), bits(host[k])), k
    assert d["best"] == host["best"]
    assert np.array_equal(d["match_idx"].cpu().numpy(), np.concatenate(host["match_idx"]))
    assert np.array_equal(bits(d["match_w"].cpu().numpy()), bits(np.concatenate(host["match_w"])))

    opt = LinearICPOptimizer(device=0)
    opt.setMetric(1)
    opt.setNbOfIterations(12)
    opt.setMatchingMaxDistance(0.003)
    out = opt.estimatePoseBatchIndexed(sources, targets, poses)
    with capi.Context(0) as ctx:
        ctx.set_config(opt.config())
        want = ctx.estimate_pose_batch_indexed(sources, targets, poses)
    assert len(out) == len(sources) and all(np.array_equal(a, b) for a, b in zip(out, want["poses"]))
    assert [e is None for e in opt.last_error] == [s == capi.OK for s in want["status"]]
