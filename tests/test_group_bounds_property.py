"""CPU property test of the pruning rule of the group search (csrc/knn.cu: GroupBounds / group_keeps): a restatement in numpy
fp32 of the two node tests, with round-to-nearest where the device rounds outwards (so the restated bounds are at most as wide as
the device's: what holds here holds there).  Claim: a box that holds a point p whose D1 distance (contract D1: fp32,
((dx*dx + dy*dy) + dz*dz), no FMA) to SOME member is <= that member's bound is never dropped -- whatever the scale of the
coordinates, the spread of the members and of their radii."""
import numpy as np
import pytest

f32 = np.float32


def d1(q, p):
    dx, dy, dz = f32(q[0] - p[0]), f32(q[1] - p[1]), f32(q[2] - p[2])
    return f32(f32(f32(dx * dx) + f32(dy * dy)) + f32(dz * dz))


def group_bounds(q, bd):
    """q [M,3] fp32 member points, bd [M] fp32 member bounds (squared distances of real points)."""
    r = (np.sqrt(bd).astype(f32) * f32(1.00001)).astype(f32)                   # device: __fmul_ru(__fsqrt_ru(bd), 1.00001f) >= this
    bl = (q - r[:, None]).astype(f32).min(0); bh = (q + r[:, None]).astype(f32).max(0)   # device: rounded outwards
    ql, qh = q.min(0), q.max(0)
    dlim = f32(f32(bd.max() * f32(1.0001)) + f32(1e-36))
    return bl, bh, ql, qh, dlim


def group_keeps(g, lo, hi):
    bl, bh, ql, qh, dlim = g
    meets = bool(np.all(lo <= bh) and np.all(hi >= bl))
    gap = np.maximum(np.maximum((lo - qh).astype(f32), (ql - hi).astype(f32)), f32(0))
    g2 = f32(f32(f32(gap[0] * gap[0]) + f32(gap[1] * gap[1])) + f32(gap[2] * gap[2]))
    return meets and not (g2 > dlim)


@pytest.mark.parametrize("scale", [1e-3, 1.0, 17.0, 4000.0])
def test_no_box_with_a_candidate_is_dropped(scale):
    rng = np.random.default_rng(int(scale * 1000) + 5)
    checked = 0
    for trial in range(400):
        m = int(rng.integers(1, 33))
        centre = rng.uniform(-scale, scale, 3)
        spread = scale * 10.0 ** rng.uniform(-4, 0)
        q = (centre + rng.normal(0, spread, size=(m, 3))).astype(f32)
        # a cloud of target points around the members, some at exactly-tying distances (mirror images), some duplicates of members
        reach = spread * 10.0 ** rng.uniform(-2, 1.5)
        pts = (centre + rng.normal(0, reach, size=(60, 3))).astype(f32)
        pts = np.concatenate([pts, (2 * q[:1] - pts[:5]).astype(f32), q[:2]])
        dist = np.array([[d1(qq, p) for p in pts] for qq in q], dtype=f32)                 # [M, P]
        # every member's bound is the distance of a real point (its previous neighbour): the k-th nearest for a random small k
        k = rng.integers(0, 4, size=m)
        bd = np.array([np.sort(dist[i])[k[i]] for i in range(m)], dtype=f32)
        g = group_bounds(q, bd)
        cand = np.where((dist <= bd[:, None]).any(0))[0]                                   # points that can change some member's answer
        for j in cand:
            # boxes of the hierarchy are exact min / max of their points: the tightest (the point alone) and looser ones around it
            for grow in (0.0, reach * 0.01, reach):
                others = pts[rng.integers(0, len(pts), 3)] if grow else pts[j][None]
                lo = np.minimum(pts[j], others.min(0)).astype(f32) - f32(grow) * (grow == reach)
                hi = np.maximum(pts[j], others.max(0)).astype(f32) + f32(grow) * (grow == reach)
                assert group_keeps(g, lo.astype(f32), hi.astype(f32)), (scale, trial, j, grow)
                checked += 1
    assert checked > 2000


def test_far_boxes_are_dropped():
    """The rule prunes: a box farther from every member than the largest radius goes."""
    q = np.array([[0, 0, 0], [0.1, 0.05, 0]], f32)
    bd = np.array([1.0, 1.21], f32)                                                        # radii 1.0 and 1.1
    g = group_bounds(q, bd)
    assert group_keeps(g, np.array([0.9, 0, 0], f32), np.array([1.5, 0.2, 0.2], f32))
    assert not group_keeps(g, np.array([1.3, 0, 0], f32), np.array([1.5, 0.2, 0.2], f32))      # beyond the balls' box
    assert not group_keeps(g, np.array([0.9, 0.9, 0.9], f32), np.array([1.0, 1.0, 1.0], f32))  # inside the box of the balls, outside every ball
