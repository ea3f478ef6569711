"""Row N (the Ceres Levenberg-Marquardt driver) pinned against something that was NOT written from the same memory.

oracle/ref_shim/ceres/ceres.h and oracle/icp_oracle.c:orc_solve_lm are two restatements of Ceres' trust-region loop by one author,
so their bit-for-bit agreement only proves self-consistency.  Independent here:
  * the residuals are the reference's OWN functors (constraints.h:9-143, compiled in place, evaluated through oracle/_ref), assembled
    exactly as CeresICPOptimizer::prepareConstraints* adds them (ICPOptimizer.h:363-482: a PointToPoint block per match, plus a
    PointToPlane / Symmetric block for the plane / symmetric metric);
  * the minimiser is scipy's MINPACK Levenberg-Marquardt (`least_squares(method="lm")`) run to machine precision.
What Ceres documents: Solve stops when the relative cost decrease falls below function_tolerance = 1e-6 (and the reference keeps the
defaults, ICPOptimizer.h:352-360), so its answer is not the minimiser but lies within that tolerance of it.  The tests therefore
require   cost(x_LM) <= cost(x*) * (1 + 2e-6)   and   |x_LM - x*| <= 5e-4   for the oracle's LM, for the reference build's LM and for
the device's LM.  What stays unpinned: Ceres' exact iterate sequence (radius schedule, accept / reject decisions) when it does NOT
converge within max_num_iterations = 10 -- no Ceres binary exists in this environment to compare with.

Where the reference build is absent the residuals are the functors' closed forms in oracle/oracle_as_ref.py, checked against the
build by tests/test_oracle_vs_reference.py::test_oracle_as_ref_answers_like_the_reference where it exists and against scipy's
axis-angle rotation in every checkout (tests/test_reference_golden.py).  They are numpy, not the oracle's C jets, so the oracle's and
the device's LM reaching their minimum still pins two independent statements of the functors against each other; the reference
build's own LM is then not run.
"""
import numpy as np
import pytest
from scipy.optimize import least_squares
from scipy.spatial.transform import Rotation

from icp_variants_b200 import synth
from oracle import oracle as O
from oracle import oracle_as_ref, ref

R = ref if ref.available() else oracle_as_ref


def _problem(metric):
    src, tgt, _, _ = synth.load_bunny()
    cfg = O.Config(metric=metric, minimizer=1, max_distance_sq=0.0003, n_iterations=1)
    m, tp, tn = O.match_pipeline(cfg, np.eye(4, dtype=np.float32), src.points, src.normals, src.colors, tgt.points, tgt.normals, tgt.colors,
                                 return_transformed=True)
    keep = np.nonzero(m["idx"] >= 0)[0]

    def residuals(x):
        out = []
        for i in keep:
            j = m["idx"][i]; w = float(m["weight"][i])
            out.extend(R.residuals(0, x, tp[i], tgt.points[j], tn[i], tgt.normals[j], w))                 # ICPOptimizer.h:383-388
            if metric:
                out.extend(np.atleast_1d(R.residuals(metric, x, tp[i], tgt.points[j], tn[i], tgt.normals[j], w)))   # :425-430 / :471-476
        return np.asarray(out, np.float64)

    sol = least_squares(residuals, np.zeros(6), method="lm", xtol=1e-15, ftol=1e-15, gtol=1e-15)
    return src, tgt, m, tp, tn, residuals, sol


def _cost(residuals, x):
    r = residuals(x)
    return 0.5 * float(r @ r)


def _x_from_pose(pose):
    return np.r_[Rotation.from_matrix(pose[:3, :3].astype(np.float64)).as_rotvec(), pose[:3, 3].astype(np.float64)]


@pytest.mark.parametrize("metric", [0, 1, 2])
def test_oracle_and_reference_lm_reach_the_independent_minimum(metric):
    src, tgt, m, tp, tn, residuals, sol = _problem(metric)
    rc, x, pose_o, n_lm = O.solve_lm(metric, tp, tn, tgt.points, tgt.normals, m, max_iterations=10)
    assert rc == 0 and 1 <= n_lm <= 10
    assert _cost(residuals, x) <= sol.cost * (1 + 2e-6)
    assert np.abs(x - sol.x).max() <= 5e-4
    assert _cost(residuals, np.zeros(6)) > 1.2 * sol.cost                      # the problem is not trivial
    if not ref.available():
        return
    # the reference's CeresICPOptimizer (over the Ceres stand-in), one outer iteration from the identity
    n, pose_r, _ = R.estimate_pose(1, metric, src.points, src.normals, src.colors, tgt.points, tgt.normals, tgt.colors, src.points[:4], tgt.points[:4],
                                   n_iterations=1, max_distance_sq=0.0003)
    assert n == 1
    assert _cost(residuals, _x_from_pose(pose_r)) <= sol.cost * (1 + 2e-6)


@pytest.mark.gpu
@pytest.mark.parametrize("metric", [0, 1, 2])
def test_device_lm_reaches_the_independent_minimum(metric):
    from icp_variants_b200 import capi
    src, tgt, m, tp, tn, residuals, sol = _problem(metric)
    cfg = capi.default_config()
    cfg.metric, cfg.minimizer, cfg.n_iterations, cfg.max_distance_sq, cfg.nn_algorithm = metric, 1, 1, 0.0003, 2
    with capi.Context(0) as ctx:
        ctx.set_config(cfg)
        ctx.set_target(tgt.points, tgt.normals, tgt.colors)
        ctx.set_source(src.points, src.normals, src.colors)
        pose, _, n_it = ctx.estimate_pose()
    assert n_it == 1
    x = _x_from_pose(pose)
    assert _cost(residuals, x) <= sol.cost * (1 + 2e-6)
    assert np.abs(x - sol.x).max() <= 5e-4
