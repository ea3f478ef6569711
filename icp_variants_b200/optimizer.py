"""Host-side mirror of the reference's operator interface for the registration path, in Python on
top of the icp_gpu_* C ABI (the C++14 mirror is include/icp_b200/*.h).  Names, argument meaning and
defaults follow the reference so that tests read like its drivers (main.cpp / experiment.cpp):

    ICPOptimizer / LinearICPOptimizer / CeresICPOptimizer   ICPOptimizer.h:27-175, :489, :181
    NearestNeighborSearch{Flann,BruteForce,Projective}      NearestNeighbor.h:12-36, :104, :42, :317
    Match                                                   NearestNeighbor.h:7-10
    TimeMeasure / ConvergenceMeasure                        TimeMeasure.h:7-62, ConvergenceMeasure.h:15-184

Everything computes on the device; nothing here falls back to the CPU.
"""
from __future__ import annotations

from dataclasses import dataclass, field

import numpy as np

from . import capi
from .synth import Cloud as PointCloud  # points / normals / colours AoS, PointCloud.h

# selection.h:8, weighting.h:8
SELECT_ALL, RANDOM_SAMPLING = 0, 1
CONSTANT_WEIGHTING, DISTANCES_WEIGHTING, NORMALS_WEIGHTING, COLORS_WEIGHTING = 0, 1, 2, 3
MAX_DISTANCE = 0.005  # NearestNeighbor.h:5

MATCH_DTYPE = np.dtype([("idx", np.int32), ("weight", np.float32)])  # Match{int idx; float weight}


@dataclass
class TimeMeasure:
    """TimeMeasure.h:7-62 -- the accumulators the loop fills, here from CUDA events (seconds)."""
    selectionTime: float = 0.0
    matchingTime: float = 0.0
    weighingTime: float = 0.0
    rejectionTime: float = 0.0
    solverTime: float = 0.0
    convergenceTime: float = 0.0
    indexTime: float = 0.0
    nIterations: int = 0

    def calculateIterationTime(self):
        n = max(self.nIterations, 1)
        return {k: getattr(self, k) / n for k in ("selectionTime", "matchingTime", "weighingTime", "rejectionTime", "solverTime")}


@dataclass
class ConvergenceMeasure:
    """ConvergenceMeasure.h:15-66: RMSE over known correspondences after each iteration
    (recordAlignmentError is fed the per-iteration pose, ICPOptimizer.h:629-631)."""
    sourceCorrespondences: np.ndarray | None = None   # [M,3]
    targetCorrespondences: np.ndarray | None = None   # [M,3]
    rmseErrors: list = field(default_factory=list)
    runBenchmark: bool = False                        # ConvergenceMeasure.h:32: also the Fontana benchmark error (:104-151)
    groundTruthPose: np.ndarray | None = None         # instead of the arrays: every source point under this pose (main.cpp:300-307)
    benchmarkErrors: list = field(default_factory=list)

    def recordAlignmentError(self, pose):
        if self.sourceCorrespondences is None:
            return
        p = np.asarray(pose, np.float32)
        s = np.asarray(self.sourceCorrespondences, np.float32)
        t = (s @ p[:3, :3].T + p[:3, 3]).astype(np.float32)
        d = t - np.asarray(self.targetCorrespondences, np.float32)
        ok = np.isfinite(t).all(1) & np.isfinite(self.targetCorrespondences).all(1)
        sq = ((d[ok, 0] * d[ok, 0] + d[ok, 1] * d[ok, 1]) + d[ok, 2] * d[ok, 2]).astype(np.float32)
        self.rmseErrors.append(float(np.sqrt(np.float32(sq.sum(dtype=np.float32) / np.float32(max(int(ok.sum()), 1))))))


class NearestNeighborSearch:
    """NearestNeighbor.h:12-36.  buildIndex uploads the target and builds the device grid;
    queryMatches returns Match records for already-transformed query points."""
    _matching = 0
    _nn_algorithm = 0

    def __init__(self, device: int = 0, ctx: capi.Context | None = None):
        self._ctx = ctx or capi.Context(device)
        self.m_maxDistance = MAX_DISTANCE
        self._have_index = False
        self._colors = False

    def setMatchingMaxDistance(self, maxDistance: float):
        self.m_maxDistance = float(maxDistance)

    def setCameraParams(self, depthIntrinsics, width, height):
        self._ctx.set_camera(depthIntrinsics, width, height)

    def buildIndex(self, targetPoints, targetColors=None):
        self._ctx.set_target(targetPoints, None, targetColors)
        self._have_index = True
        self._colors = targetColors is not None

    def queryMatches(self, transformedPoints, transformedColors=None):
        if not self._have_index:
            # NearestNeighbor.h:144-147: message + empty result
            print("FLANN index needs to be build before querying any matches.")
            return np.empty(0, MATCH_DTYPE)
        if self._colors != (transformedColors is not None):
            print("Index and query dimensionality do not agree.")   # :148-152
            return np.empty(0, MATCH_DTYPE)
        cfg = capi.default_config()
        cfg.matching = self._matching
        cfg.nn_algorithm = self._nn_algorithm
        cfg.max_distance_sq = self.m_maxDistance
        cfg.rejection = 0
        cfg.weighting = CONSTANT_WEIGHTING
        cfg.color_icp = int(self._colors)
        self._ctx.set_config(cfg)
        self._ctx.set_source(transformedPoints, None, transformedColors)
        idx, w = self._ctx.query_matches(np.eye(4, dtype=np.float32))
        out = np.empty(len(idx), MATCH_DTYPE)
        out["idx"], out["weight"] = idx, w
        return out


class NearestNeighborSearchFlann(NearestNeighborSearch):
    """NearestNeighbor.h:104-314.  The reference's FLANN search is approximate (1 randomized kd-tree,
    16 checks); this returns the exact nearest neighbour (ties to the lowest index)."""
    _nn_algorithm = 2   # grid


class NearestNeighborSearchBruteForce(NearestNeighborSearch):
    """NearestNeighbor.h:42-98 as written: candidates compared on the rounded norm, m_maxDistance taken as a plain distance (:93)."""
    _nn_algorithm = 3


class NearestNeighborSearchProjective(NearestNeighborSearch):
    """NearestNeighbor.h:317-444."""
    _matching = 1


class ICPOptimizer:
    """ICPOptimizer.h:27-175: options + estimatePose.  `minimizer` is fixed by the subclass."""
    _minimizer = 0

    def __init__(self, device: int = 0, ctx: capi.Context | None = None):
        self._ctx = ctx or capi.Context(device)
        # constructor defaults, ICPOptimizer.h:29-31
        self.metric, self.selectionMethod, self.rejectionMethod, self.weightingMethod = 0, SELECT_ALL, 1, CONSTANT_WEIGHTING
        self.m_nIterations, self.matchingMethod, self.maxDistance = 20, 0, 0.0003
        # The reference keeps two distances apart: the matcher's own threshold (NearestNeighborSearch::m_maxDistance, MAX_DISTANCE
        # until setMatchingMaxDistance, and again after every setMatchingMethod, which re-creates the matcher, ICPOptimizer.h:71-78)
        # and ICPOptimizer::maxDistance (0.0003 until setMatchingMaxDistance), which only WeightingMethod sees (:220,:528).
        self.matcherMaxDistance = MAX_DISTANCE
        self.colorICP, self.multiResolutionICP = False, False
        self.proba = 1.0
        self.seed = 0                 # the reference seeds from std::random_device (selection.h:76-79)
        self.selection_rng = 0        # 0 mt19937 (reference-compatible), 1 device stream
        self.nn_algorithm = 0         # 0 auto, 1 brute force, 2 tiled grid search, 3 per-query tree search
        self.use_graph = True
        self.pyramid_mode = 0         # 0 the reference's stride pyramid, 1 voxel levels (extension)
        self.early_stop = (0.0, 0.0)  # extension: (radians, metres) below which an applied increment ends the loop; 0 = run all iterations
        self.m_timeMeasure: TimeMeasure | None = None
        self.m_convergenceMeasure: ConvergenceMeasure | None = None
        self._camera = None
        self.last_error: str | None = None

    def setMatchingMaxDistance(self, maxDistance):
        self.matcherMaxDistance = float(maxDistance)      # m_nearestNeighborSearch->setMatchingMaxDistance, ICPOptimizer.h:42
        self.maxDistance = float(maxDistance)             # :43

    def setMetric(self, metric):
        self.metric = int(metric)

    def enableMultiResolution(self, enable):
        self.multiResolutionICP = bool(enable)

    def enableColorICP(self, colorICP):
        self.colorICP = bool(colorICP)

    def setSelectionMethod(self, selectionMethod, proba=1.0):
        self.selectionMethod, self.proba = int(selectionMethod), float(proba)

    def setRejectionMethod(self, rejectionMethod):
        self.rejectionMethod = int(rejectionMethod)

    def setWeightingMethod(self, weightingMethod):
        self.weightingMethod = int(weightingMethod)

    def setMatchingMethod(self, matchingMethod):
        # ICPOptimizer.h:71-78 re-creates the matcher, which resets its max distance to MAX_DISTANCE
        self.matchingMethod = int(matchingMethod)
        self.matcherMaxDistance = MAX_DISTANCE            # the weighting distance keeps its value

    def setCameraParamsMatchingMethod(self, depthIntrinsics, width, height):
        self._camera = (np.asarray(depthIntrinsics, np.float32), int(width), int(height))

    def setNbOfIterations(self, nIterations):
        self.m_nIterations = int(nIterations)

    def setTimeMeasure(self, timeMeasure: TimeMeasure):
        self.m_timeMeasure = timeMeasure

    def setConvergenceMeasure(self, convergenceMeasure: ConvergenceMeasure):
        self.m_convergenceMeasure = convergenceMeasure

    def config(self) -> capi.Config:
        c = capi.default_config()
        c.metric, c.minimizer, c.matching = self.metric, self._minimizer, self.matchingMethod
        c.selection, c.proba, c.seed, c.selection_rng = self.selectionMethod, self.proba, self.seed & 0xFFFFFFFF, self.selection_rng
        c.weighting, c.rejection, c.max_distance_sq = self.weightingMethod, self.rejectionMethod, self.matcherMaxDistance
        c.weight_max_distance_sq = self.maxDistance
        c.color_icp, c.multires, c.n_iterations = int(self.colorICP), int(self.multiResolutionICP), self.m_nIterations
        c.nn_algorithm, c.use_graph, c.pyramid_mode = self.nn_algorithm, int(self.use_graph), self.pyramid_mode
        c.early_stop_rotation, c.early_stop_translation = float(self.early_stop[0]), float(self.early_stop[1])
        return c

    def setTarget(self, target: PointCloud):
        """buildIndex (ICPOptimizer.h:532-535): upload the target and build the device grid."""
        self._ctx.set_target(target.points, target.normals, target.colors)

    def setSource(self, source: PointCloud):
        self._ctx.set_source(source.points, source.normals, source.colors)

    def estimatePose(self, source: PointCloud | None, target: PointCloud | None, initialPose, calculateRMSE=True):
        """ICPOptimizer.h:140.  Returns the estimated pose (the reference writes it into initialPose).
        Passing None for a cloud reuses the one already resident on the device."""
        self._ctx.set_config(self.config())
        if self._camera is not None:
            self._ctx.set_camera(*self._camera)
        if target is not None:
            self.setTarget(target)
        if source is not None:
            self.setSource(source)
        want_hist = calculateRMSE and self.m_convergenceMeasure is not None
        want_t = self.m_timeMeasure is not None
        self.last_error = None
        try:
            res = self._ctx.estimate_pose(initialPose, want_history=want_hist, timings=want_t)
        except capi.IcpGpuError as e:
            if e.code not in (capi.E_NO_MATCHES, capi.E_NUMERIC):
                raise
            # the reference hangs in ASSERT here (Eigen.h:9); the drop-in keeps the last good pose
            self.last_error = str(e)
            return e.pose
        pose, hist, n_it = res[:3]
        if want_t:
            tm, t = self.m_timeMeasure, res[3]
            tm.matchingTime += t.matching_ms * 1e-3
            tm.solverTime += t.solver_ms * 1e-3
            tm.convergenceTime += t.total_ms * 1e-3
            tm.indexTime += t.index_ms * 1e-3
            tm.nIterations = n_it
        cm = self.m_convergenceMeasure
        if want_hist and n_it > 0 and (cm.sourceCorrespondences is not None or cm.groundTruthPose is not None):
            # recordAlignmentError after every iteration (ICPOptimizer.h:629-631), evaluated on the device from the pose history
            if cm.groundTruthPose is not None:
                self._ctx.set_correspondences_pose(cm.groundTruthPose)
            else:
                self._ctx.set_correspondences(cm.sourceCorrespondences, cm.targetCorrespondences)
            rmse, bench = self._ctx.convergence_errors(benchmark=cm.runBenchmark)
            cm.rmseErrors.extend(float(r) for r in rmse)
            if cm.runBenchmark:
                cm.benchmarkErrors.extend(float(b) for b in bench)
        return pose

    def estimatePoseBatch(self, sources, targets, initialPoses=None):
        """Many independent small registrations with this optimizer's configuration (one thread block per pair; targets of at
        most capi.BATCH_MAX_TARGET points): either minimiser, multi-resolution and mt19937 selection included.  Returns the list
        of estimated poses.  last_error becomes a list with one entry per pair: None, or the message of a pair that stopped
        without a surviving match or on a singular system (that pair's pose is its last good one, as estimatePose returns it)."""
        poses, n_it, status = self._ctx.estimate_pose_batch_configs([self.config()], np.zeros(len(sources), np.int32), sources, targets,
                                                                    initialPoses)
        self.last_error = []
        for s, n in zip(status, n_it):
            if s == capi.OK:
                self.last_error.append(None)
            elif s == capi.E_NO_MATCHES:
                self.last_error.append(f"iteration {n} had no surviving correspondence")
            else:
                self.last_error.append(f"iteration {n}: singular / non-finite normal equations")
        return list(poses)

    def estimateNormals(self, points, k: int = 5, viewpoint=None):
        """PointCloud(pcl cloud) (PointCloud.h:41-76): k-NN PCA normals of a cloud, computed on the device.  The cloud is
        indexed as the target to do so (set the registration's target afterwards if it is another cloud)."""
        pts = np.ascontiguousarray(points, np.float32)
        self._ctx.set_target(pts, None, None)
        return self._ctx.target_normals(k, viewpoint, n=len(pts))

    def setTargetFromDepth(self, depthMap, colorFrame, depthIntrinsics, depthExtrinsics=None, keepOriginalSize=False, downsampleFactor=1,
                           maxDistance=0.1):
        """PointCloud(depthMap, colorFrame, ...) (PointCloud.h:78-165) built on the device and indexed as the target
        (reconstructRoom, main.cpp:202-206); returns the number of points."""
        return self._ctx.cloud_from_depth(depthMap, colorFrame, depthIntrinsics, depthExtrinsics, keepOriginalSize, downsampleFactor,
                                          maxDistance, role=0, download=False)

    def setSourceFromDepth(self, depthMap, colorFrame, depthIntrinsics, depthExtrinsics=None, keepOriginalSize=False, downsampleFactor=1,
                           maxDistance=0.1):
        """The same for the source frame (main.cpp:295-298)."""
        return self._ctx.cloud_from_depth(depthMap, colorFrame, depthIntrinsics, depthExtrinsics, keepOriginalSize, downsampleFactor,
                                          maxDistance, role=1, download=False)


class LinearICPOptimizer(ICPOptimizer):
    """ICPOptimizer.h:489-899."""
    _minimizer = 0


class CeresICPOptimizer(ICPOptimizer):
    """ICPOptimizer.h:181-483 (Levenberg-Marquardt, <= 10 inner iterations)."""
    _minimizer = 1
