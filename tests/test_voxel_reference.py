"""The C restatement of voxel-grid downsampling (tests/voxel_reference.c, DESIGN.md section 4 rows V1-V5) against a separate one in
numpy and Python floats: float32 products, np.floor, np.lexsort, and sequential Python-float (fp64) sums in ascending index."""
import math

import os
import sys

import numpy as np
import pytest

from icp_variants_b200 import synth

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import voxel_reference as vref  # noqa: E402


def restated(pts, voxel_size, nrm=None, rgba=None, off=None):
    pts = np.asarray(pts, np.float32)
    off = np.array([0, len(pts)], np.int64) if off is None else np.asarray(off, np.int64)
    inv = np.float32(1.0) / np.float32(voxel_size)
    P, N, Cc, O = [], [], [], [0]
    for b in range(len(off) - 1):
        s, e = int(off[b]), int(off[b + 1])
        ids = s + np.nonzero(np.isfinite(pts[s:e]).all(axis=1))[0]
        v = np.floor(pts[ids] * inv).astype(np.int64)                      # float32 product, then floor
        order = np.lexsort((ids, v[:, 0], v[:, 1], v[:, 2]))               # (iz, iy, ix), then the index
        ids, v = ids[order], v[order]
        j = 0
        while j < len(ids):
            k = j + 1
            while k < len(ids) and (v[k] == v[j]).all():
                k += 1
            run = ids[j:k]
            sums = [0.0, 0.0, 0.0]
            for i in run:
                for a in range(3):
                    sums[a] += float(pts[i, a])
            P.append([np.float32(sums[a] / len(run)) for a in range(3)])
            if nrm is not None:
                q, any_ = [0.0, 0.0, 0.0], False
                for i in run:
                    if np.isfinite(nrm[i]).all():
                        any_ = True
                        for a in range(3):
                            q[a] += float(nrm[i, a])
                ln = math.sqrt(q[0] * q[0] + q[1] * q[1] + q[2] * q[2])
                N.append([np.float32(q[a] / ln) for a in range(3)] if any_ and ln != 0.0 else [-np.inf] * 3)
            if rgba is not None:
                n = len(run)
                Cc.append([(2 * int(rgba[run, ch].astype(np.int64).sum()) + n) // (2 * n) for ch in range(4)])
            j = k
        O.append(len(P))
    P = np.array(P, np.float32).reshape(-1, 3)
    N = np.array(N, np.float32).reshape(-1, 3) if nrm is not None else None
    Cc = np.array(Cc, np.uint8).reshape(-1, 4) if rgba is not None else None
    return P, N, Cc, np.array(O, np.int64)


def check(pts, size, nrm=None, rgba=None, off=None):
    got = vref.voxel_downsample(pts, size, nrm=nrm, rgba=rgba, off=off)
    want = restated(pts, size, nrm=nrm, rgba=rgba, off=off)
    for g, w in zip(got, want):
        assert (g is None) == (w is None)
        if g is not None:
            assert g.shape == w.shape and g.tobytes() == w.tobytes()
    return got


def test_bunny(bunny):
    src = bunny[0]
    p, n, c, o = check(src.points, 0.004, nrm=src.normals, rgba=src.colors)
    assert 0 < o[-1] < len(src.points)


def test_small_eth_scan_with_colours(small_eth_pair):
    tgt = small_eth_pair[1]
    col = synth.procedural_colors(tgt.points)
    for size in (0.05, 0.2):
        check(tgt.points, size, nrm=tgt.normals, rgba=col)


def test_points_on_faces_negative_coordinates_and_duplicates():
    g = np.arange(-8, 9, dtype=np.float32) * np.float32(0.25)             # exact multiples of the voxel edge: on the faces
    pts = np.stack(np.meshgrid(g, g[::2], g[::3], indexing="ij"), -1).reshape(-1, 3)
    pts = np.concatenate([pts, pts[:50], np.array([[-0.0, 0.0, -0.0], [0.0, -0.0, 0.0]], np.float32)])
    rng = np.random.default_rng(3)
    nrm = rng.normal(size=pts.shape).astype(np.float32)
    col = rng.integers(0, 256, size=(len(pts), 4)).astype(np.uint8)
    p, _, _, o = check(pts, 0.25, nrm=nrm, rgba=col)
    assert o[-1] < len(pts)


def test_non_finite_points_and_normals():
    rng = np.random.default_rng(5)
    pts = rng.uniform(-1.0, 1.0, size=(3000, 3)).astype(np.float32)
    nrm = rng.normal(size=pts.shape).astype(np.float32)
    pts[::7, 0] = np.nan
    pts[3::11, 2] = -np.inf
    pts[5::13, 1] = np.inf
    nrm[::3, 1] = np.nan
    nrm[1::5, 0] = -np.inf
    col = rng.integers(0, 256, size=(len(pts), 4)).astype(np.uint8)
    check(pts, 0.3, nrm=nrm, rgba=col)
    # a voxel whose normals cancel, one whose normals are all non-finite: MINF
    pts2 = np.array([[0.1, 0.1, 0.1], [0.2, 0.2, 0.2], [1.1, 0.1, 0.1], [1.2, 0.1, 0.1]], np.float32)
    nrm2 = np.array([[0, 0, 1], [0, 0, -1], [np.nan, 0, 0], [0, np.inf, 0]], np.float32)
    _, n2, _, _ = check(pts2, 1.0, nrm=nrm2)
    assert np.all(n2 == -np.inf)


def test_colours_round_half_up():
    pts = np.zeros((4, 3), np.float32)
    col = np.array([[0, 1, 255, 2], [1, 2, 254, 3], [0, 0, 0, 0], [0, 0, 0, 0]], np.uint8)
    _, _, c, _ = check(pts[:2], 1.0, rgba=col[:2])
    assert c.tolist() == [[1, 2, 255, 3]]                                 # (2*1 + 2) // 4 = 1: half rounds up


def test_batch_with_empty_clouds_equals_clouds_alone(small_eth_pair):
    src, tgt, _ = small_eth_pair
    clouds = [src.points[:4000], np.zeros((0, 3), np.float32), tgt.points[1000:7000], np.zeros((0, 3), np.float32), src.points[5000:5001]]
    off = np.zeros(len(clouds) + 1, np.int64)
    off[1:] = np.cumsum([len(c) for c in clouds])
    p, _, _, o = check(np.concatenate(clouds), 0.1, off=off)
    for b, c in enumerate(clouds):
        pb, _, _, ob = vref.voxel_downsample(c, 0.1)
        assert p[o[b]:o[b + 1]].tobytes() == pb.tobytes() and ob[-1] == o[b + 1] - o[b]


def test_one_voxel_and_own_voxels():
    rng = np.random.default_rng(9)
    pts = rng.uniform(0.0, 0.99, size=(500, 3)).astype(np.float32)
    _, _, _, o = check(pts, 1.0)
    assert o[-1] == 1
    _, _, _, o = check(pts, 1e-4)
    assert o[-1] == 500


def test_index_outside_int32_is_refused():
    with pytest.raises(ValueError, match="cloud 1"):
        vref.voxel_downsample(np.array([[0, 0, 0], [3e9, 0, 0]], np.float32), 1.0, off=np.array([0, 1, 2]))
