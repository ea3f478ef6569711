"""Oracle self-consistency for stage 2 (matching): exact kd-tree == literal brute force
(NearestNeighbor.h:81-97 tie rule), and both agree with an independent exact search (scipy)."""
import numpy as np
import pytest
from scipy.spatial import cKDTree

from oracle import oracle as O


def _rand_cloud(rng, n, quant=None):
    p = rng.uniform(-1, 1, size=(n, 3)).astype(np.float32)
    if quant:
        p = (np.round(p * quant) / quant).astype(np.float32)
    return p


@pytest.mark.parametrize("quant", [None, 4, 16])
def test_kdtree_equals_brute_3d(quant):
    rng = np.random.default_rng(0)
    tgt = _rand_cloud(rng, 3000, quant)
    qry = _rand_cloud(rng, 2000, quant)
    for max_d2 in (1e-3, 0.05, 10.0):
        a = O.knn_brute(tgt, qry, max_d2)
        b = O.KdTree(tgt).query(qry, max_d2)
        assert np.array_equal(a["idx"], b["idx"])
        assert np.array_equal(a["weight"], b["weight"])


def test_ties_go_to_lowest_index():
    tgt = np.array([[1, 0, 0], [-1, 0, 0], [0, 1, 0], [0, -1, 0], [1, 0, 0]], np.float32)
    qry = np.array([[0, 0, 0], [1, 0, 0], [0.5, 0.5, 0]], np.float32)
    for m in (O.knn_brute(tgt, qry, 10.0), O.KdTree(tgt).query(qry, 10.0)):
        assert m["idx"].tolist() == [0, 0, 0]
    # duplicates of the whole target: every answer must be < n
    rng = np.random.default_rng(1)
    base = _rand_cloud(rng, 500)
    tgt = np.concatenate([base, base, base])
    qry = _rand_cloud(rng, 700)
    m = O.KdTree(tgt).query(qry, 10.0)
    assert (m["idx"] < 500).all() and (m["idx"] >= 0).all()
    assert np.array_equal(m["idx"], O.knn_brute(tgt, qry, 10.0)["idx"])


def test_threshold_is_squared_and_inclusive():
    tgt = np.array([[0, 0, 0]], np.float32)
    qry = np.array([[0.5, 0, 0], [0.50001, 0, 0]], np.float32)
    m = O.knn_brute(tgt, qry, 0.25)          # NearestNeighbor.h:182 '<=' on the squared distance
    assert m["idx"].tolist() == [0, -1] and m["weight"].tolist() == [1.0, 0.0]


def test_against_scipy_exact_search():
    rng = np.random.default_rng(2)
    tgt = _rand_cloud(rng, 5000)
    qry = _rand_cloud(rng, 3000)
    m = O.KdTree(tgt).query(qry, 100.0)
    d, j = cKDTree(tgt.astype(np.float64)).query(qry.astype(np.float64))
    # continuous data: the fp32 arg-min equals the fp64 arg-min except at ~1 ulp near-ties
    same = m["idx"] == j
    assert same.mean() > 0.999
    dd = np.linalg.norm(tgt[m["idx"][~same]].astype(np.float64) - qry[~same], axis=1)
    assert np.allclose(dd, d[~same], rtol=1e-6)


def test_non_finite_points():
    tgt = np.array([[0, 0, 0], [-np.inf, -np.inf, -np.inf], [1, 1, 1]], np.float32)
    qry = np.array([[0.9, 1, 1], [np.nan, 0, 0], [-np.inf, -np.inf, -np.inf]], np.float32)
    for m in (O.knn_brute(tgt, qry, 10.0), O.KdTree(tgt).query(qry, 10.0)):
        assert m["idx"].tolist() == [2, -1, -1]


def test_6d_colour_search():
    rng = np.random.default_rng(3)
    tgt = _rand_cloud(rng, 2000, 8)
    qry = _rand_cloud(rng, 1500, 8)
    tc = rng.integers(0, 256, size=(2000, 4), dtype=np.uint8)
    qc = rng.integers(0, 256, size=(1500, 4), dtype=np.uint8)
    a = O.knn_brute(tgt, qry, 10.0, tc, qc)
    b = O.KdTree(tgt, tc).query(qry, 10.0, qc)
    assert np.array_equal(a["idx"], b["idx"])
    # independent restatement of NearestNeighbor.h:245-255 in numpy (fp64 arg-min over 6-D features)
    s = np.float32(1.0) * (np.float32(1) / np.float32(255))
    tf = np.concatenate([tgt, (s * tc[:, :3].astype(np.float32)).astype(np.float32)], 1).astype(np.float64)
    qf = np.concatenate([qry, (s * qc[:, :3].astype(np.float32)).astype(np.float32)], 1).astype(np.float64)
    d, j = cKDTree(tf).query(qf)
    diff = a["idx"] != j
    # quantised positions + colours can tie in fp64 only by exact duplicates; allow equal-distance alternates
    da = np.linalg.norm(tf[a["idx"]] - qf, axis=1)
    assert np.allclose(da, d, rtol=1e-5, atol=1e-7), diff.sum()


def test_packed_key_order_equals_lexicographic_distance_index_order():
    """The grid search kernels compare candidates as ONE unsigned 64-bit key bits(d2) << 32 | idx (search.cuh: better_key;
    knn.cu: thread_scan_leaf).  That is the (d2, idx) lexicographic order of contract D2 for every non-negative fp32 distance --
    +0, denormals, FLT_MAX, +inf -- and puts NaN distances after every number, as the strict comparisons of
    NearestNeighbor.h:81-97 do."""
    rng = np.random.default_rng(11)
    special = np.array([0.0, 1e-45, 1.1754944e-38, 1.0, 10.0, 3.4028235e38, np.inf], np.float32)
    d = np.concatenate([special, rng.random(2000).astype(np.float32) * 5.0, rng.choice(special, 500)]).astype(np.float32)
    idx = rng.integers(0, 2**31 - 1, size=len(d)).astype(np.int64)
    idx[: len(special)] = [0, 2**31 - 2, 5, 5, 0, 1, 7]
    key = (d.view(np.uint32).astype(np.uint64) << np.uint64(32)) | idx.astype(np.uint64)
    i, j = rng.integers(0, len(d), 20000), rng.integers(0, len(d), 20000)
    lex = (d[i] < d[j]) | ((d[i] == d[j]) & (idx[i] < idx[j]))
    assert np.array_equal(key[i] < key[j], lex)
    nan_key = (np.array([np.nan], np.float32).view(np.uint32).astype(np.uint64) << np.uint64(32))
    assert (nan_key[0] > key).all()          # a NaN distance never wins
    # the initial bound (min(max_d2, FLT_MAX), INT_MAX) loses exactly to the candidates the reference accepts: d2 <= max_d2
    init = (np.array([10.0], np.float32).view(np.uint32).astype(np.uint64) << np.uint64(32)) | np.uint64(2**31 - 1)
    assert np.array_equal(key < init[0], (d <= np.float32(10.0)) & ~((d == np.float32(10.0)) & (idx >= 2**31 - 1)))
