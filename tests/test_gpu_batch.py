"""GPU tests of the batched registration (icp_gpu_estimate_pose_batch, csrc/batch.cu): one thread block per pair runs
the pair's whole loop.  Every pair must follow the oracle's trajectory (free-running, 1e-5 rad / 1e-5 m at every
iteration), agree with the single-pair path, pick the brute-force scan's correspondences bit for bit, stop on its own
and leave its neighbours and the context's own registration alone."""
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
    return rot_angle(pa, pb) <= tol and float(np.linalg.norm(pa[:3, 3].astype(np.float64) - pb[:3, 3])) <= tol


def perturbation(seed, max_angle=0.02, max_trans=0.002):
    """A seeded small rigid motion (bunny scale: ~0.1 m)."""
    rng = np.random.default_rng(seed)
    axis = rng.normal(size=3); axis /= np.linalg.norm(axis)
    a = rng.uniform(0.0, max_angle)
    K = np.array([[0, -axis[2], axis[1]], [axis[2], 0, -axis[0]], [-axis[1], axis[0], 0]])
    P = np.eye(4)
    P[:3, :3] = np.eye(3) + np.sin(a) * K + (1 - np.cos(a)) * K @ K
    P[:3, 3] = rng.uniform(-max_trans, max_trans, 3)
    return P.astype(np.float32)


def config(metric=1, weighting=0, rejection=1, n_iterations=20, max_d2=0.0003, **kw):
    c = capi.default_config()
    c.metric, c.weighting, c.rejection, c.n_iterations, c.max_distance_sq = metric, weighting, rejection, n_iterations, max_d2
    for k, v in kw.items():
        setattr(c, k, v)
    return c


def oracle(cfg, src, tgt, init):
    ocfg = orc.Config(metric=cfg.metric, weighting=cfg.weighting, rejection=cfg.rejection, max_distance_sq=cfg.max_distance_sq,
                      n_iterations=cfg.n_iterations)
    return orc.estimate_pose(ocfg, src.points, src.normals, src.colors, tgt.points, tgt.normals, tgt.colors, init_pose=init)


def assert_follows_oracle(cfg, src, tgt, init, pose, hist, n_it, status, what=""):
    rc, opose, ohist, _ = oracle(cfg, src, tgt, init)
    assert rc == 0 and status == capi.OK, (what, rc, status)
    assert n_it == len(ohist), (what, n_it, len(ohist))
    for k in range(n_it):
        assert pose_close(hist[k], ohist[k]), f"{what} iteration {k}: rot {rot_angle(hist[k], ohist[k]):.2e} trans {np.linalg.norm(hist[k][:3, 3] - ohist[k][:3, 3]):.2e}"
    assert np.array_equal(pose, hist[n_it - 1])
    assert not hist[n_it:].any()


@pytest.fixture(scope="module")
def ctx():
    c = capi.Context(0)
    yield c
    c.close()


@pytest.fixture(scope="module")
def inits():
    return np.stack([perturbation(100 + b) for b in range(8)])


# ----------------------------------------------------------------------------- 1. free-running parity with the oracle
@pytest.mark.parametrize("metric", [0, 1, 2])
@pytest.mark.parametrize("weighting", [0, 1, 2])
@pytest.mark.parametrize("rejection", [0, 1])
def test_free_running_parity(ctx, bunny, inits, metric, weighting, rejection):
    src, tgt, _, _ = bunny
    cfg = config(metric, weighting, rejection)
    ctx.set_config(cfg)
    poses, n_it, status, hist = ctx.estimate_pose_batch([src] * 8, [tgt] * 8, inits, want_history=True)
    for b in range(8):
        assert_follows_oracle(cfg, src, tgt, inits[b], poses[b], hist[b], n_it[b], status[b], f"pair {b}")


# ----------------------------------------------------------------------------- 2. batch equals single
@pytest.mark.parametrize("metric", [0, 1, 2])
def test_batch_equals_single(ctx, bunny, inits, metric):
    src, tgt, _, _ = bunny
    cfg = config(metric, weighting=1)
    ctx.set_config(cfg)
    poses, n_it, status = ctx.estimate_pose_batch([src] * 8, [tgt] * 8, inits)
    ctx.set_target(tgt.points, tgt.normals, tgt.colors)
    ctx.set_source(src.points, src.normals, src.colors)
    for b in range(8):
        pose, _, n = ctx.estimate_pose(inits[b], want_history=False)
        assert status[b] == capi.OK and n_it[b] == n
        assert pose_close(poses[b], pose), f"pair {b}: rot {rot_angle(poses[b], pose):.2e} trans {np.linalg.norm(poses[b][:3, 3] - pose[:3, 3]):.2e}"


# ----------------------------------------------------------------------------- 3. bit-exact correspondences
def test_correspondences_bit_exact_on_ties_duplicates_and_nonfinite(ctx):
    """One query per pair, all against one quantised target with exact ties, duplicates (with opposite normals, so that
    picking the higher index of a duplicate is rejected) and non-finite points.  With a single match the point-to-point
    step is the pure translation t[idx] - s, so every pair's pose names the target point it matched; a rejected or missing
    match is ICP_GPU_E_NO_MATCHES with the start pose."""
    rng = np.random.default_rng(7)
    tgt = (rng.integers(0, 8, size=(2000, 3)) * 0.25).astype(np.float32)
    tgt_n = np.tile(np.array([[0, 0, 1]], np.float32), (len(tgt), 1))
    tgt[100:200] = tgt[0:100]                    # duplicates with higher indices ...
    tgt_n[100:150] = [0, 0, -1]                  # ... half of them rejected by the normal test
    tgt_n[0:25] = [0, 0, -1]; tgt_n[100:125] = [0, 0, 1]   # and lower-index copies rejected where the higher one is not
    tgt[300] = [np.inf, 0, 0]; tgt[301] = [np.nan, 1, 1]; tgt[302] = [-np.inf, -np.inf, -np.inf]
    qry = (rng.integers(-2, 10, size=(600, 3)) * 0.25 + 0.125 * rng.integers(0, 2, size=(600, 3))).astype(np.float32)
    qry[:100] = tgt[:100]                        # exactly on the duplicated points
    qry[5] = [np.nan, 0, 0]; qry[6] = [-np.inf, -np.inf, -np.inf]
    qry_n = np.tile(np.array([[0, 0, 1]], np.float32), (len(qry), 1))
    ocfg = orc.Config(metric=0, rejection=1, max_distance_sq=1.0, n_iterations=1, nn_mode=0)
    om = orc.match_pipeline(ocfg, np.eye(4, dtype=np.float32), qry, qry_n, None, tgt, tgt_n, None)
    assert (om["idx"] >= 0).sum() > 400 and (om["idx"] < 0).sum() > 20
    ctx.set_config(config(metric=0, rejection=1, n_iterations=1, max_d2=1.0))
    srcs = [synth.Cloud(qry[i:i + 1], qry_n[i:i + 1], None) for i in range(len(qry))]
    poses, n_it, status = ctx.estimate_pose_batch(srcs, [synth.Cloud(tgt, tgt_n, None)] * len(qry))
    for i in range(len(qry)):
        j = om["idx"][i]
        if j < 0:
            assert status[i] == capi.E_NO_MATCHES and n_it[i] == 0 and np.array_equal(poses[i], np.eye(4, dtype=np.float32)), i
        else:
            assert status[i] == capi.OK and n_it[i] == 1, i
            assert np.array_equal(poses[i][:3, 3], (tgt[j].astype(np.float64) - qry[i]).astype(np.float32)), (i, j, poses[i][:3, 3])
            assert np.array_equal(poses[i][:3, :3], np.eye(3, dtype=np.float32)), i


@pytest.mark.parametrize("metric", [0, 1, 2])
def test_teacher_forced_single_iteration(ctx, bunny, metric):
    """One iteration from every pose of the oracle's trajectory = the oracle's own step on its own matches."""
    src, tgt, _, _ = bunny
    cfg = config(metric, n_iterations=20)
    rc, _, ohist, _ = oracle(cfg, src, tgt, perturbation(5))
    assert rc == 0
    starts = np.concatenate([perturbation(5)[None], ohist[:-1]])
    cfg1 = config(metric, n_iterations=1)
    ctx.set_config(cfg1)
    poses, n_it, status = ctx.estimate_pose_batch([src] * len(starts), [tgt] * len(starts), starts)
    for k, start in enumerate(starts):
        rc, opose, _, _ = oracle(cfg1, src, tgt, start)
        assert rc == 0 and status[k] == capi.OK and n_it[k] == 1
        assert pose_close(poses[k], opose, 1e-6), f"start {k}: rot {rot_angle(poses[k], opose):.2e} trans {np.linalg.norm(poses[k][:3, 3] - opose[:3, 3]):.2e}"


# ----------------------------------------------------------------------------- 4. heterogeneous batch
def padded_target(tgt, n):
    """The bunny target followed by copies shifted 5 m and more away (never matched), n points in all."""
    reps = [tgt.points] + [tgt.points + np.float32(5.0 * k) for k in range(1, n // len(tgt.points) + 2)]
    nrm = np.tile(tgt.normals, (len(reps), 1))
    return synth.Cloud(np.concatenate(reps)[:n].copy(), nrm[:n].copy(), None)


def test_heterogeneous_batch(ctx, bunny, inits):
    src, tgt, _, _ = bunny
    empty = synth.Cloud(np.zeros((0, 3), np.float32), np.zeros((0, 3), np.float32), None)
    far = synth.Cloud(src.points + np.float32(10.0), src.normals, None)
    half = synth.Cloud(src.points[::2].copy(), src.normals[::2].copy(), None)
    big = padded_target(tgt, capi.BATCH_MAX_TARGET)
    pairs = [(src, tgt), (empty, tgt), (src, empty), (far, tgt), (half, tgt), (src, big), (src, tgt)]
    init = np.stack([inits[b % len(inits)] for b in range(len(pairs))])
    init[5] = init[0]
    cfg = config(metric=2)
    ctx.set_config(cfg)
    poses, n_it, status, hist = ctx.estimate_pose_batch([p[0] for p in pairs], [p[1] for p in pairs], init, want_history=True)
    for b in (0, 4, 5, 6):
        assert_follows_oracle(cfg, pairs[b][0], pairs[b][1], init[b], poses[b], hist[b], n_it[b], status[b], f"pair {b}")
    for b in (1, 2, 3):
        assert status[b] == capi.E_NO_MATCHES and n_it[b] == 0, b
        assert np.array_equal(poses[b], init[b]) and not hist[b].any(), b
    # the pair with the full target registers like the bunny alone, bit for bit (the copies are never matched)
    assert np.array_equal(poses[5], poses[0]) and np.array_equal(hist[5], hist[0])
    with pytest.raises(capi.IcpGpuError) as e:
        ctx.estimate_pose_batch([src, src], [tgt, padded_target(tgt, capi.BATCH_MAX_TARGET + 1)])
    assert e.value.code == capi.E_ARG and "8193" in str(e.value)


# ----------------------------------------------------------------------------- 5. determinism
def test_deterministic(ctx, bunny, inits):
    src, tgt, _, _ = bunny
    ctx.set_config(config(metric=2, weighting=2))
    B = len(inits)
    init = inits.copy(); init[B - 1] = init[0]
    a = ctx.estimate_pose_batch([src] * B, [tgt] * B, init, want_history=True)
    b = ctx.estimate_pose_batch([src] * B, [tgt] * B, init, want_history=True)
    for x, y in zip(a, b):
        assert np.array_equal(x, y)
    assert np.array_equal(a[0][0], a[0][B - 1]) and np.array_equal(a[3][0], a[3][B - 1])


# ----------------------------------------------------------------------------- 6. refusals
@pytest.mark.parametrize("field,value", [("minimizer", 1), ("multires", 1), ("matching", 1), ("color_icp", 1),
                                         ("selection", 1), ("nn_algorithm", 3)])
def test_refused_configurations(ctx, bunny, field, value):
    src, tgt, _, _ = bunny
    cfg = config(metric=1, selection_rng=0, proba=0.5)
    setattr(cfg, field, value)
    ctx.set_config(cfg)
    with pytest.raises(capi.IcpGpuError) as e:
        ctx.estimate_pose_batch([src], [tgt])
    assert e.value.code == capi.E_ARG


def _raw_batch(ctx, src_off, tgt_off, n_src, n_tgt):
    B = len(src_off) - 1
    sp = np.zeros((max(n_src, 1), 3), np.float32); tp = np.zeros((max(n_tgt, 1), 3), np.float32)
    so, to = np.asarray(src_off, np.int64), np.asarray(tgt_off, np.int64)
    pin = np.tile(np.eye(4, dtype=np.float32).reshape(16), (B, 1)); pout = np.zeros_like(pin)
    n_it = np.zeros(B, np.int32); st = np.zeros(B, np.int32)
    p = capi._ptr
    return capi.lib().icp_gpu_estimate_pose_batch(ctx._h, B, p(sp), None, p(so), p(tp), None, p(to), p(pin), p(pout), p(n_it), p(st), None)


def test_refused_offsets_and_pending_registration(ctx, bunny):
    torch = pytest.importorskip("torch")
    src, tgt, _, _ = bunny
    ctx.set_config(config(metric=1))
    assert _raw_batch(ctx, [0, 5, 3], [0, 4, 8], 5, 8) == capi.E_ARG                  # not monotone
    assert _raw_batch(ctx, [1, 5], [0, 4], 5, 4) == capi.E_ARG                        # not starting at 0
    assert _raw_batch(ctx, [0, 5], [0, 4], 5, 4) == capi.OK
    d = torch.device("cuda", 0)
    sp = torch.zeros((5, 3), device=d); tp = torch.zeros((4, 3), device=d)
    with pytest.raises(capi.IcpGpuError) as e:                                        # offsets that do not match the arrays
        ctx.estimate_pose_batch_dev(sp, torch.tensor([0, 6], device=d), tp, torch.tensor([0, 4], device=d))
    assert e.value.code == capi.E_ARG
    # the context's own registration: the same pose before and after a batch; a batch while it is pending is refused
    ctx.set_target(tgt.points, tgt.normals, tgt.colors)
    ctx.set_source(src.points, src.normals, src.colors)
    before, _, _ = ctx.estimate_pose(perturbation(1), want_history=False)
    ctx.estimate_pose_async(perturbation(1))
    with pytest.raises(capi.IcpGpuError) as e:
        ctx.estimate_pose_batch([src], [tgt])
    assert e.value.code == capi.E_STATE
    pending, _ = ctx.estimate_pose_finish()
    ctx.estimate_pose_batch([src.points[::3], src], [tgt, tgt.points[::2]])
    after, _, _ = ctx.estimate_pose(perturbation(1), want_history=False)
    assert np.array_equal(before, pending) and np.array_equal(before, after)


# ----------------------------------------------------------------------------- 7. device selection stream
def test_device_random_selection(ctx, bunny, inits):
    """Each pair selects with the single-pair path's device stream (hash of the pair-local index): about p of the points,
    the same pose as icp_gpu_estimate_pose, and it converges on the bunny."""
    src, tgt, gs, gt = bunny
    cfg = config(metric=2, selection=1, proba=0.5, seed=3, selection_rng=1)
    ctx.set_config(cfg)
    init = np.concatenate([np.eye(4, dtype=np.float32)[None], inits[:3]])
    poses, n_it, status = ctx.estimate_pose_batch([src] * 4, [tgt] * 4, init)
    ctx.set_target(tgt.points, tgt.normals, tgt.colors)
    ctx.set_source(src.points, src.normals, src.colors)
    for b in range(4):
        pose, _, n = ctx.estimate_pose(init[b], want_history=False)
        frac = ctx.stats().n_queries / (n * len(src))
        assert 0.45 < frac < 0.55
        assert status[b] == capi.OK and n_it[b] == n == 20
        assert pose_close(poses[b], pose)
        assert orc.rmse(poses[b], src.points[gs], tgt.points[gt]) < 1e-3


def test_optimizer_estimate_pose_batch(bunny, inits):
    src, tgt, _, _ = bunny
    opt = LinearICPOptimizer(device=0)
    opt.setMetric(1)
    opt.setMatchingMaxDistance(0.0003)
    far = synth.Cloud(src.points + np.float32(10.0), src.normals, None)
    poses = opt.estimatePoseBatch([src, far], [tgt, tgt], inits[:2])
    assert opt.last_error[0] is None and "no surviving correspondence" in opt.last_error[1]
    single = opt.estimatePose(src, tgt, inits[0], calculateRMSE=False)
    assert pose_close(poses[0], single) and np.array_equal(poses[1], inits[1])


# ----------------------------------------------------------------------------- 8. torch plumbing
def test_torch_dev_form_equals_host_form(ctx, bunny, inits):
    torch = pytest.importorskip("torch")
    src, tgt, _, _ = bunny
    ctx.set_config(config(metric=2, weighting=1))
    srcs = [src, synth.Cloud(src.points[::2].copy(), src.normals[::2].copy(), None), src]
    tgts = [tgt, tgt, synth.Cloud(tgt.points[::3].copy(), tgt.normals[::3].copy(), None)]
    host = ctx.estimate_pose_batch(srcs, tgts, inits[:3], want_history=True)
    d = torch.device("cuda", 0)
    sp, sn, so = capi._concat_clouds(srcs)
    tp, tn, to = capi._concat_clouds(tgts)
    t = lambda a: torch.from_numpy(a).to(d)
    dev = ctx.estimate_pose_batch_dev(t(sp), t(so), t(tp), t(to), t(sn), t(tn), t(inits[:3]), want_history=True)
    for h, g in zip(host, dev):
        assert g.is_cuda and np.array_equal(h, g.cpu().numpy())
