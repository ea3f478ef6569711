"""The slice of oracle/ref.py's interface that the device-vs-reference tests call, answered by the oracle (oracle/icp_oracle.c).

TEST INFRASTRUCTURE ONLY.  The tests compare the device against oracle/ref.py (the reference's own headers compiled in place)
where that build exists, and against this module elsewhere.  The oracle is pinned to the reference build by
tests/test_oracle_vs_reference.py (bit-exact matching, weighting, rejection, transforms and depth constructor; 1e-5 rad / 1e-5 m
poses; the LM path bit-exact) and, on every machine, to the reference's stored outputs by tests/test_reference_golden.py.
Return values and argument orders are those of oracle/ref.py.
"""
from __future__ import annotations

import numpy as np

from oracle import oracle as O

transform_points = O.transform_points
transform_normals = O.transform_normals
cloud_from_depth = O.cloud_from_depth

MAX_DISTANCE_SQ = 0.005        # the matcher's distance after setMatchingMethod (NearestNeighbor.h:5,35, ICPOptimizer.h:71-78)
DEFAULT_MAX_DISTANCE_SQ = 0.0003   # ICPOptimizer::maxDistance when setMatchingMaxDistance is never called (ICPOptimizer.h:29-31)


def _pair(m):
    return m["idx"].copy(), m["weight"].copy()


def _matches(idx, w):
    m = np.empty(len(idx), O.MATCH_DTYPE)
    m["idx"], m["weight"] = idx, w
    return m


def knn_flann(tgt, qry, max_d2, tgt_rgba=None, qry_rgba=None):
    return _pair(O.knn_brute(tgt, qry, max_d2, tgt_rgba, qry_rgba))


def knn_brute(tgt, qry, max_d):
    return _pair(O.knn_brute_norm(tgt, qry, max_d))


def projective(tgt, width, height, fx, fy, cx, cy, qry, max_d2):
    return _pair(O.projective(tgt, width, height, fx, fy, cx, cy, qry, max_d2))


def apply_weights(method, max_d2, sp, sn, sc, tp, tn, tc, idx, w):
    return _pair(O.apply_weights(method, max_d2, sp, sn, sc, tp, tn, tc, _matches(idx, w)))


def prune(sn, tn, idx, w):
    return _pair(O.prune(sn, tn, _matches(idx, w)))


def solve_linear(metric, s, d, ns, nt, w):
    if metric == 0:
        return O.solve_p2p(s, d, w)
    if metric == 1:
        return O.solve_p2plane(s, d, nt, w)
    return O.solve_symmetric(s, d, ns, nt, w)


def _rotate(x, p):
    """ceres::AngleAxisRotatePoint: Rodrigues, first order below theta^2 = eps."""
    th = np.linalg.norm(x[:3])
    K = np.array([[0, -x[2], x[1]], [x[2], 0, -x[0]], [-x[1], x[0], 0]])
    if th * th <= np.finfo(float).eps:
        return (np.eye(3) + K) @ p, np.eye(3) + K
    Rm = np.eye(3) + np.sin(th) / th * K + (1 - np.cos(th)) / th ** 2 * K @ K
    return Rm @ p, Rm


def residuals(kind, x, s, d, ns, nt, w):
    """The functors of constraints.h:9-143 in closed form: 0 point-to-point (weight 0.1), 1 point-to-plane, 2 symmetric."""
    x = np.asarray(x, np.float64)
    s, d, ns, nt = (np.asarray(v, np.float32).astype(np.float64) for v in (s, d, ns, nt))
    w = np.float64(np.float32(w))
    y, Rm = _rotate(x, s)
    y = y + x[3:]
    if kind == 0:
        return np.float64(np.float32(0.1)) * w * (y - d)
    if kind == 1:
        return np.array([w * (nt @ (y - d))])
    return np.array([w * ((nt + ns) @ (y - Rm.T @ d))])


def estimate_pose(minimizer, metric, src, src_n, src_c, tgt, tgt_n, tgt_c, gt_src, gt_ref, *, n_iterations=20, max_distance_sq=0.0003,
                  selection=0, proba=1.0, seed=0, weighting=0, rejection=1, matching=0, color_icp=False, multires=False,
                  camera=None, init_pose=None, setter_order=0):
    """(n_iterations_executed | -2, pose, rmse history) as oracle/ref.py returns them.  setter_order 1 / 2: the matcher keeps
    MAX_DISTANCE, the weighting max_distance_sq / the constructor's default."""
    match_d2, weight_d2 = max_distance_sq, 0.0
    if setter_order == 1:
        match_d2, weight_d2 = MAX_DISTANCE_SQ, max_distance_sq
    elif setter_order == 2:
        match_d2, weight_d2 = MAX_DISTANCE_SQ, DEFAULT_MAX_DISTANCE_SQ
    cam = {}
    if camera is not None:
        fx, fy, cx, cy, width, height = camera
        cam = dict(fx=float(fx), fy=float(fy), cx=float(cx), cy=float(cy), width=int(width), height=int(height))
    cfg = O.Config(metric=metric, minimizer=minimizer, matching=matching, selection=selection, proba=proba, seed=seed, weighting=weighting,
                   rejection=rejection, max_distance_sq=match_d2, weight_max_distance_sq=weight_d2, color_icp=bool(color_icp),
                   multires=bool(multires), n_iterations=n_iterations, **cam)
    rc, pose, hist, _ = O.estimate_pose(cfg, src, src_n, src_c, tgt, tgt_n, tgt_c, init_pose=init_pose)
    rmse = np.array([O.rmse(h, gt_src, gt_ref) for h in hist], np.float32)
    return (len(hist) if rc == 0 else -2), pose, rmse
