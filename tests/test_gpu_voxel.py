"""GPU tests of voxel-grid downsampling (icp_gpu_voxel_downsample[_dev], csrc/voxel.cu and csrc/voxel_api.cu): points, normals, colours
and offsets bit for bit against the CPU restatement tests/voxel_reference.c (DESIGN.md section 4, V1-V5) on the bunny, the full ETH-shaped scan at several sizes and
edge cases; keys wider than one 32-bit word; batches against clouds filtered alone, in any order and with a launch count independent
of the number of clouds; the TARGET / SOURCE / ONLY roles; the device form; refusals."""

import os
import sys

import numpy as np
import pytest

from icp_variants_b200 import capi, synth

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import voxel_reference as vref  # noqa: E402

pytestmark = pytest.mark.gpu

ONLY, TARGET, SOURCE = 2, 0, 1


@pytest.fixture(scope="module")
def ctx():
    c = capi.Context(0)
    yield c
    c.close()


def cheap_normals(pts, viewpoint):
    """Unit vectors towards the sensor: normals for the filter's arithmetic, without the seconds of a host PCA over 370k points."""
    d = (np.asarray(viewpoint, np.float64) - pts.astype(np.float64))
    return (d / np.linalg.norm(d, axis=1, keepdims=True)).astype(np.float32)


@pytest.fixture(scope="module")
def eth_scan():
    """The full ~370k-point ETH-shaped scan with textured colours."""
    room = synth.make_room(1234)
    return synth.lidar_scan(room, np.array([6.0, 4.5, 1.2]), n_sweeps=344, n_beams=1077, seed=7, colors="texture", normals_fn=cheap_normals)


def run(ctx, pts, size, nrm=None, rgba=None, off=None):
    """The host form on concatenated clouds: (points, normals, colours, offsets)."""
    pts, nrm, rgba = capi._f32(pts, 3), capi._f32(nrm, 3), capi._u8(rgba)
    off = np.array([0, len(pts)], np.int64) if off is None else np.ascontiguousarray(off, np.int64)
    return ctx._voxel_host(pts, nrm, rgba, off, size, ONLY)


def same(got, want):
    for g, w in zip(got, want):
        assert (g is None) == (w is None)
        if g is not None:
            assert g.shape == w.shape and g.tobytes() == w.tobytes()


def check(ctx, pts, size, nrm=None, rgba=None, off=None):
    got = run(ctx, pts, size, nrm, rgba, off)
    same(got, vref.voxel_downsample(pts, size, nrm=nrm, rgba=rgba, off=off))
    return got


def test_bunny(ctx, bunny):
    src = bunny[0]
    for size in (0.002, 0.004, 0.01):
        _, _, _, o = check(ctx, src.points, size, src.normals, src.colors)
        assert 0 < o[-1] < len(src.points)


@pytest.mark.parametrize("size", [0.02, 0.05, 0.1, 0.2])
def test_full_eth_scan(ctx, eth_scan, size):
    assert len(eth_scan.points) > 300_000
    check(ctx, eth_scan.points, size, eth_scan.normals, eth_scan.colors)


def test_duplicates_faces_and_negative_zero(ctx):
    g = np.arange(-8, 9, dtype=np.float32) * np.float32(0.25)
    pts = np.stack(np.meshgrid(g, g[::2], g[::3], indexing="ij"), -1).reshape(-1, 3)
    pts = np.concatenate([pts, pts[:50], np.array([[-0.0, 0.0, -0.0], [0.0, -0.0, 0.0]], np.float32)])
    rng = np.random.default_rng(3)
    check(ctx, pts, 0.25, rng.normal(size=pts.shape).astype(np.float32), rng.integers(0, 256, size=(len(pts), 4)).astype(np.uint8))


def test_non_finite_points_and_normals(ctx):
    rng = np.random.default_rng(5)
    pts = rng.uniform(-1.0, 1.0, size=(30000, 3)).astype(np.float32)
    nrm = rng.normal(size=pts.shape).astype(np.float32)
    pts[::7, 0] = np.nan
    pts[3::11, 2] = -np.inf
    pts[5::13, 1] = np.inf
    nrm[::3, 1] = np.nan
    nrm[1::5, 0] = -np.inf
    check(ctx, pts, 0.1, nrm, rng.integers(0, 256, size=(len(pts), 4)).astype(np.uint8))
    # only non-finite points: no voxel
    _, _, _, o = check(ctx, np.full((100, 3), np.nan, np.float32), 0.1)
    assert o.tolist() == [0, 0]


def test_cancelling_normals(ctx):
    pts = np.array([[0.1, 0.1, 0.1], [0.2, 0.2, 0.2], [1.1, 0.1, 0.1], [1.2, 0.1, 0.1], [2.5, 0.5, 0.5]], np.float32)
    nrm = np.array([[0, 0, 1], [0, 0, -1], [np.nan, 0, 0], [0, np.inf, 0], [0, 3, 4]], np.float32)
    _, n, _, _ = check(ctx, pts, 1.0, nrm)
    assert np.all(n[:2] == -np.inf) and n[2].tolist() == [0.0, np.float32(0.6), np.float32(0.8)]


def test_one_voxel_and_own_voxels(ctx):
    rng = np.random.default_rng(9)
    pts = rng.uniform(0.0, 0.99, size=(20000, 3)).astype(np.float32)
    col = rng.integers(0, 256, size=(len(pts), 4)).astype(np.uint8)
    _, _, _, o = check(ctx, pts, 1.0, rgba=col)
    assert o[-1] == 1
    _, _, _, o = check(ctx, pts, 1e-5, rgba=col)
    assert o[-1] == len(pts)


def test_empty_clouds(ctx):
    e = np.zeros((0, 3), np.float32)
    p, n, c, o = check(ctx, e, 0.1, e, np.zeros((0, 4), np.uint8))
    assert len(p) == 0 and o.tolist() == [0, 0]
    _, _, _, o = check(ctx, e, 0.1, off=np.zeros(5, np.int64))
    assert o.tolist() == [0] * 5


def test_wide_keys(ctx):
    """About 2^15 voxels per axis: 45 key bits, two words.  2^21 voxels per axis on two clouds: 64 bits, three words.  One voxel more
    is refused and names the cloud."""
    rng = np.random.default_rng(11)
    pts = rng.uniform(0.0, 2.0 ** 15 * 0.01, size=(200000, 3)).astype(np.float32)
    pts[::4] = pts[1::4] + np.float32(0.001)                               # shared voxels
    check(ctx, pts, 0.01, rgba=rng.integers(0, 256, size=(len(pts), 4)).astype(np.uint8))
    edge = np.float32(2.0 ** 21 - 0.5)
    a = np.array([[0.5, 0.5, 0.5], [edge, edge, edge], [edge, 0.5, 7.5], [0.5, edge, 0.5], [0.7, 0.5, 0.5]], np.float32)
    b = -a[::-1]
    _, _, _, o = check(ctx, np.concatenate([a, b]), 1.0, off=[0, len(a), 2 * len(a)])
    assert o.tolist() == [0, 4, 8]
    wide = np.concatenate([a, [[2.0 ** 21 + 0.5, 0.5, 0.5]]]).astype(np.float32)
    with pytest.raises(capi.IcpGpuError, match="cloud 1 spans 2097153 voxels on x") as e:
        run(ctx, np.concatenate([a, wide]), 1.0, off=[0, len(a), len(a) + len(wide)])
    assert e.value.code == capi.E_ARG
    check(ctx, a, 1.0)                                                      # still usable


def mixed_batch():
    bunny = synth.load_bunny()[0]
    room = synth.make_room(1234)
    scan = synth.lidar_scan(room, np.array([6.0, 4.5, 1.2]), n_sweeps=120, n_beams=400, seed=3, colors="texture", normals_fn=cheap_normals)
    rng = np.random.default_rng(21)
    clouds = []
    for b in range(64):
        k = b % 4
        if k == 0:
            clouds.append(synth.Cloud(np.zeros((0, 3), np.float32), np.zeros((0, 3), np.float32), np.zeros((0, 4), np.uint8)))
        elif k == 1:
            s = int(rng.integers(0, len(bunny.points) // 2))
            n = int(rng.integers(1, len(bunny.points) - s))
            clouds.append(synth.Cloud(bunny.points[s:s + n], bunny.normals[s:s + n], bunny.colors[s:s + n]))
        else:
            s = int(rng.integers(0, len(scan.points) - 9000))
            n = int(rng.integers(1, 9000))
            clouds.append(synth.Cloud(scan.points[s:s + n], scan.normals[s:s + n], scan.colors[s:s + n]))
    return clouds


def test_batch_equals_clouds_alone_in_any_order(ctx):
    clouds = mixed_batch()
    xyz, n3, c4, off = capi._concat_clouds_rgba(clouds)
    got = check(ctx, xyz, 0.01, n3, c4, off)
    batch = ctx.voxel_downsample_batch(clouds, 0.01)
    for b, cl in enumerate(clouds):
        alone = ctx.voxel_downsample(cl.points, 0.01, nrm=cl.normals, rgba=cl.colors)
        same(batch[b], alone)
        same(batch[b], (got[0][got[3][b]:got[3][b + 1]], got[1][got[3][b]:got[3][b + 1]], got[2][got[3][b]:got[3][b + 1]]))
    perm = np.random.default_rng(5).permutation(len(clouds))
    shuffled = ctx.voxel_downsample_batch([clouds[i] for i in perm], 0.01)
    for j, i in enumerate(perm):
        same(shuffled[j], batch[i])


def launches(ctx, f):
    before = ctx.stats().n_kernel_launches
    f()
    return ctx.stats().n_kernel_launches - before


def test_launches_do_not_grow_with_the_batch(ctx):
    """One cloud spanning 2^8 voxels per axis and 64 clouds spanning 2^6 each: 24-bit keys both (the cloud index takes 6), so the same
    sort; the launches are the same."""
    rng = np.random.default_rng(13)
    one = rng.uniform(0.0, 255.9, size=(100000, 3)).astype(np.float32)
    one[:2] = [[0, 0, 0], [255.5, 255.5, 255.5]]
    many = []
    for b in range(64):
        c = rng.uniform(0.0, 63.9, size=(1500, 3)).astype(np.float32) + np.float32(100 * b)
        c[:2] = [[100 * b, 100 * b, 100 * b], [100 * b + 63.5] * 3]
        many.append(c)
    off = np.zeros(65, np.int64)
    off[1:] = np.cumsum([len(c) for c in many])
    n1 = launches(ctx, lambda: run(ctx, one, 1.0))
    n64 = launches(ctx, lambda: run(ctx, np.concatenate(many), 1.0, off=off))
    assert n1 == n64 > 0


def config():
    c = capi.default_config()
    c.metric, c.n_iterations, c.max_distance_sq = 1, 15, 0.01
    return c


@pytest.mark.parametrize("role", [TARGET, SOURCE])
def test_roles_set_the_cloud(small_eth_pair, role):
    src, tgt, _ = small_eth_pair
    cloud = tgt if role == TARGET else src
    pose0 = np.eye(4, dtype=np.float32)
    with capi.Context(0) as a, capi.Context(0) as b:
        for c in (a, b):
            c.set_config(config())
        if role == TARGET:
            a.set_source(src.points, src.normals)
            p, n, col = a.voxel_downsample(cloud.points, 0.05, nrm=cloud.normals, rgba=cloud.colors, role=TARGET)
            b.set_source(src.points, src.normals)
            b.set_target(p, n, col)
        else:
            a.set_target(tgt.points, tgt.normals)
            p, n, col = a.voxel_downsample(cloud.points, 0.05, nrm=cloud.normals, rgba=cloud.colors, role=SOURCE)
            b.set_target(tgt.points, tgt.normals)
            b.set_source(p, n, col)
        same((p, n, col), vref.voxel_downsample(cloud.points, 0.05, nrm=cloud.normals, rgba=cloud.colors)[:3])
        ia, wa = a.query_matches(pose0)
        ib, wb = b.query_matches(pose0)
        assert ia.tobytes() == ib.tobytes() and wa.tobytes() == wb.tobytes()
        ra, rb = a.estimate_pose(pose0), b.estimate_pose(pose0)
        assert ra[0].tobytes() == rb[0].tobytes() and ra[1].tobytes() == rb[1].tobytes() and ra[2] == rb[2]


def test_role_only_leaves_the_context(small_eth_pair, eth_scan):
    src, tgt, _ = small_eth_pair
    with capi.Context(0) as a, capi.Context(0) as b:
        for c in (a, b):
            c.set_config(config())
            c.set_target(tgt.points, tgt.normals)
            c.set_source(src.points, src.normals)
        first = a.estimate_pose(), b.estimate_pose()
        assert first[0][0].tobytes() == first[1][0].tobytes()
        a.voxel_downsample(eth_scan.points, 0.05, nrm=eth_scan.normals, rgba=eth_scan.colors, role=ONLY)
        a.voxel_downsample_batch([src, tgt], 0.02)
        ra, rb = a.estimate_pose(), b.estimate_pose()
        assert ra[0].tobytes() == rb[0].tobytes() and ra[1].tobytes() == rb[1].tobytes() and ra[2] == rb[2]
        assert a.query_matches(ra[0])[0].tobytes() == b.query_matches(rb[0])[0].tobytes()


def test_dev_form_and_repeat(ctx, eth_scan):
    torch = pytest.importorskip("torch")
    dev = torch.device("cuda", 0)
    clouds = mixed_batch()[:16]
    xyz, n3, c4, off = capi._concat_clouds_rgba(clouds)
    host = run(ctx, xyz, 0.02, n3, c4, off)
    p, n, c, o = ctx.voxel_downsample_dev(torch.from_numpy(xyz).to(dev), torch.from_numpy(off).to(dev), 0.02,
                                          nrm=torch.from_numpy(n3).to(dev), rgba=torch.from_numpy(c4).to(dev))
    same((p.cpu().numpy(), n.cpu().numpy(), c.cpu().numpy(), o.cpu().numpy()), host)
    again = run(ctx, xyz, 0.02, n3, c4, off)
    same(again, host)
    big = run(ctx, eth_scan.points, 0.05, eth_scan.normals, eth_scan.colors)
    same(run(ctx, eth_scan.points, 0.05, eth_scan.normals, eth_scan.colors), big)
    # without normals and colours, and the dev form as the context's target
    # without normals and colours
    p, n, c, o = ctx.voxel_downsample_dev(torch.from_numpy(xyz).to(dev), torch.from_numpy(off).to(dev), 0.02)
    assert n is None and c is None
    plain = run(ctx, xyz, 0.02, off=off)
    same((p.cpu().numpy(), o.cpu().numpy()), (plain[0], plain[3]))


def raw(ctx, n_clouds, xyz, off, size=0.1, role=ONLY, nrm=None, rgba=None, xyz_out=True, nrm_out=None, rgba_out=None, off_out=True):
    cap = max(len(xyz) if xyz is not None else 1, 1)
    po = np.empty((cap, 3), np.float32) if xyz_out else None
    oo = np.zeros(max(n_clouds + 1, 1), np.int64) if off_out else None
    return capi.lib().icp_gpu_voxel_downsample(ctx._h, n_clouds, capi._ptr(xyz), capi._ptr(nrm), capi._ptr(rgba), capi._ptr(off), float(size),
                                               role, capi._ptr(po), capi._ptr(nrm_out), capi._ptr(rgba_out), capi._ptr(oo))


def test_refusals_leave_the_context_usable(ctx, small_eth_pair):
    src, tgt, _ = small_eth_pair
    x = np.ascontiguousarray(src.points[:1000])
    nr = np.ascontiguousarray(src.normals[:1000])
    o1 = np.array([0, 1000], np.int64)
    buf = np.empty((1000, 3), np.float32)
    cases = [
        dict(n_clouds=-1, xyz=x, off=o1),
        dict(n_clouds=1, xyz=None, off=o1),
        dict(n_clouds=1, xyz=x, off=None),
        dict(n_clouds=1, xyz=x, off=o1, xyz_out=False),
        dict(n_clouds=1, xyz=x, off=o1, off_out=False),
        dict(n_clouds=1, xyz=x, off=o1, nrm_out=buf),
        dict(n_clouds=1, xyz=x, off=o1, rgba_out=np.empty((1000, 4), np.uint8)),
        dict(n_clouds=1, xyz=x, off=np.array([1, 1000], np.int64)),
        dict(n_clouds=2, xyz=x, off=np.array([0, 600, 500], np.int64)),
        dict(n_clouds=1, xyz=x, off=o1, size=0.0),
        dict(n_clouds=1, xyz=x, off=o1, size=-0.1),
        dict(n_clouds=1, xyz=x, off=o1, size=float("nan")),
        dict(n_clouds=1, xyz=x, off=o1, size=float("inf")),
        dict(n_clouds=1, xyz=x, off=o1, role=3),
        dict(n_clouds=1, xyz=x, off=o1, role=-1),
        dict(n_clouds=2, xyz=x, off=np.array([0, 500, 1000], np.int64), role=TARGET),
        dict(n_clouds=0, xyz=x, off=o1, role=SOURCE),
        dict(n_clouds=1, xyz=x, off=np.array([0, 0x7fffffff // 4 + 1], np.int64)),
        dict(n_clouds=2, xyz=np.array([[0, 0, 0], [3e9, 0, 0]], np.float32), off=np.array([0, 1, 2], np.int64), size=1.0),
        dict(n_clouds=1, xyz=np.array([[0, 0, 0], [0, 0, 2.0 ** 21 + 1]], np.float32), off=np.array([0, 2], np.int64), size=1.0),
    ]
    for k, case in enumerate(cases):
        assert raw(ctx, **case) == capi.E_ARG, (k, capi.lib().icp_gpu_last_error(ctx._h))
        same(run(ctx, x, 0.05, nr), vref.voxel_downsample(x, 0.05, nrm=nr))
    assert raw(ctx, 2, np.array([[0, 0, 0], [3e9, 0, 0]], np.float32), np.array([0, 1, 2], np.int64), size=1.0) == capi.E_ARG
    assert "cloud 1" in capi.lib().icp_gpu_last_error(ctx._h).decode()
    assert raw(ctx, 0, None, None) == capi.OK                              # nothing runs
    with capi.Context(0) as c:
        c.set_config(config())
        c.set_target(tgt.points, tgt.normals)
        c.set_source(src.points, src.normals)
        c.estimate_pose_async()
        assert raw(c, 1, x, o1) == capi.E_STATE
        c.estimate_pose_finish()
        same(run(c, x, 0.05, nr), vref.voxel_downsample(x, 0.05, nrm=nr))
