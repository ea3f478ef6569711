"""The CSV experiment runner (experiment.cpp:414-451) on the device path: every row of an experiment file
(Data/experiment.csv, Data/bunny_experiments.csv: expName, expType, useLinear, useMetric, matchingMethod, selectionMethod,
weightingMethod, useMultiresolution, numIterations, maxMatchingDist, samplingProba) configures an optimizer exactly as the
scenario functions of experiment.cpp do and runs it; the per-iteration RMSE goes to `<expName>_RMSE.txt`
(ConvergenceMeasure::writeRMSEToFile, ConvergenceMeasure.h:153-163).

Scenario inputs are supplied by the caller (the reference reads them from fixed paths under Data/):
    "bunny": (source Cloud, target Cloud, gt source indices, gt target indices)        experiment.cpp:22-141
    "room" : (depth frames [n,h,w], K 3x3, ground-truth poses [n,4,4] or None)           experiment.cpp:143-274
    "eth"  : list of (source Cloud, target Cloud, unchanged source points)                experiment.cpp:276-412
"""
from __future__ import annotations

import os
from dataclasses import dataclass

import numpy as np

from .optimizer import CeresICPOptimizer, ConvergenceMeasure, LinearICPOptimizer, TimeMeasure
from .sequence import alignPairs, reconstructRoom


@dataclass
class Experiment:
    expName: str
    expType: str
    useLinear: int
    useMetric: int
    matchingMethod: int
    selectionMethod: int
    weightingMethod: int
    useMultiresolution: int
    numIterations: int
    maxMatchingDist: float
    samplingProba: float


def read_experiments(path: str) -> list:
    """CSVReader::getData + the row parsing of experiment.cpp:424-437 (the first line is the header)."""
    out = []
    with open(path) as f:
        rows = [ln.rstrip("\r\n").split(",") for ln in f if ln.strip()]
    for cf in rows[1:]:
        out.append(Experiment(cf[0], cf[1], int(cf[2]), int(cf[3]), int(cf[4]), int(cf[5]), int(cf[6]), int(cf[7]), int(cf[8]), float(cf[9]), float(cf[10])))
    return out


def _optimizer(e: Experiment, device: int, seed: int, ctx=None):
    opt = (LinearICPOptimizer if e.useLinear else CeresICPOptimizer)(device=device, ctx=ctx)
    opt.seed = seed                                                  # the reference seeds from std::random_device (selection.h:76-79)
    opt.setMetric(e.useMetric)
    opt.setNbOfIterations(e.numIterations)
    return opt


def write_rmse(path: str, values):
    with open(path, "w") as f:
        for v in values:
            f.write(f"{np.float32(v):g}\n")                         # operator<<(float): 6 significant digits


def _configure_bunny(opt, e: Experiment):
    opt.setMatchingMethod(0)
    opt.setMatchingMaxDistance(e.maxMatchingDist)
    opt.setSelectionMethod(e.selectionMethod, e.samplingProba)
    opt.setWeightingMethod(e.weightingMethod)
    opt.enableMultiResolution(bool(e.useMultiresolution))


def run_experiment(e: Experiment, inputs: dict, out_dir: str = ".", device: int = 0, seed: int = 0) -> dict:
    """One row.  Returns {"pose" | "poses", "rmse", "file"}."""
    os.makedirs(out_dir, exist_ok=True)
    opt = _optimizer(e, device, seed)
    if e.expType == "bunny":                                        # experiment.cpp:22-141
        src, tgt, gs, gt = inputs["bunny"]
        _configure_bunny(opt, e)
        cm = ConvergenceMeasure(src.points[gs], tgt.points[gt]); tm = TimeMeasure()
        opt.setConvergenceMeasure(cm); opt.setTimeMeasure(tm)
        pose = opt.estimatePose(src, tgt, np.eye(4, dtype=np.float32))
        path = os.path.join(out_dir, e.expName + "_RMSE.txt")
        write_rmse(path, cm.rmseErrors)
        return {"pose": pose, "rmse": list(cm.rmseErrors), "file": path, "times": tm}
    if e.expType == "room":                                         # experiment.cpp:143-274
        frames, K, gt = inputs["room"]
        if e.matchingMethod:
            opt.setMatchingMethod(1)
        opt.setMatchingMaxDistance(e.maxMatchingDist)
        opt.setSelectionMethod(e.selectionMethod, e.samplingProba)
        opt.setWeightingMethod(e.weightingMethod)
        opt.enableMultiResolution(bool(e.useMultiresolution))
        res = reconstructRoom(opt, frames, K, groundTruthPoses=gt)
        files = []
        for i, r in enumerate(res.rmsePerIteration):
            files.append(os.path.join(out_dir, f"{e.expName}_RMSE{i}.txt"))
            write_rmse(files[-1], r)
        return {"poses": res.cameraToWorld, "rmse": res.rmsePerIteration, "file": files}
    if e.expType == "eth":                                          # experiment.cpp:276-412
        from . import capi
        opt.setMatchingMethod(0)
        opt.setMatchingMaxDistance(e.maxMatchingDist)
        opt.setSelectionMethod(e.selectionMethod, e.samplingProba)
        opt.setWeightingMethod(e.weightingMethod)
        opt.enableMultiResolution(bool(e.useMultiresolution))
        with capi.Context(device) as second:
            res = alignPairs([opt._ctx, second], inputs["eth"], opt.config(), calculateErrors=True)
        files = []
        for i, r in enumerate(res):
            files.append(os.path.join(out_dir, f"{e.expName}_{i}_RMSE.txt"))
            write_rmse(files[-1], r.rmseErrors)
        return {"poses": [r.pose for r in res], "rmse": [r.rmseErrors for r in res], "file": files}
    raise ValueError(f"unknown experiment type {e.expType!r}")


def _run_bunny_batch(exps: list, inputs: dict, out_dir: str, device: int, seed: int) -> list:
    """The "bunny" rows in one batched registration, one configuration per row (Context.estimate_pose_batch_configs); each
    row's RMSE per iteration is the device ConvergenceMeasure of its pose history."""
    from . import capi
    src, tgt, gs, gt = inputs["bunny"]
    out = []
    with capi.Context(device) as ctx:
        configs = []
        for e in exps:
            opt = _optimizer(e, device, seed, ctx=ctx)
            _configure_bunny(opt, e)
            configs.append(opt.config())
        B = len(exps)
        poses, n_it, _, hist = ctx.estimate_pose_batch_configs(configs, np.arange(B, dtype=np.int32), [src] * B, [tgt] * B,
                                                                    want_history=True)
        ctx.set_correspondences(src.points[gs], tgt.points[gt])
        for k, e in enumerate(exps):                             # a pair that stopped early keeps its last good pose, as estimatePose does
            rmse = [ctx.alignment_error(hist[k, i])[0] for i in range(n_it[k])]
            path = os.path.join(out_dir, e.expName + "_RMSE.txt")
            write_rmse(path, rmse)
            out.append({"pose": poses[k], "rmse": rmse, "file": path})
    return out


def run_experiments(path: str, inputs: dict, out_dir: str = ".", device: int = 0, seed: int = 0, batched: bool = False) -> list:
    """main() of experiment.cpp: every row of the file, in order.  batched=True: all "bunny" rows of the file run in one batched
    registration, one configuration per row; the other rows run as with batched=False."""
    exps = read_experiments(path)
    if not batched:
        return [run_experiment(e, inputs, out_dir, device, seed) for e in exps]
    os.makedirs(out_dir, exist_ok=True)
    rows = [i for i, e in enumerate(exps) if e.expType == "bunny"]
    out = [None] * len(exps)
    if rows:
        for i, r in zip(rows, _run_bunny_batch([exps[i] for i in rows], inputs, out_dir, device, seed)):
            out[i] = r
    return [r if r is not None else run_experiment(e, inputs, out_dir, device, seed) for e, r in zip(exps, out)]
