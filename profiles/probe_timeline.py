"""Timeline of ONE iteration (the 13th) of BASELINE config 2 inside the graph replay: start and end of every warp of knn_prep_kernel
and knn_bvh_kernel and of every block of reduce_kernel (%globaltimer, plain stores), written by a DIAGNOSTIC build of the library
(knn.cu / solve.cu compiled with -DICP_TIMELINE into lib/libicp_gpu_timeline.so, profiles/README.md).  Shows what the kernels' own
durations do not: ramps, tails, how many warps are resident over time and the gaps between dependent launches.
Usage: ICP_GPU_MATCH_CHUNKS=1|2 python profiles/probe_timeline.py"""
import ctypes as C
import json
import os
import sys

import numpy as np
import torch

os.environ.setdefault("ICP_GPU_LIB_NAME", "libicp_gpu_timeline.so")
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from icp_variants_b200 import capi, synth  # noqa: E402

TL_WARPS = 40960


def resident(starts, ends, t_grid):
    """Number of warps alive at each time of t_grid."""
    s = np.sort(starts); e = np.sort(ends)
    return np.searchsorted(s, t_grid, side="right") - np.searchsorted(e, t_grid, side="right")


def main():
    torch.cuda.set_device(0)
    lib = C.CDLL(capi.LIB_PATH)
    ctx = capi.Context(0)
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    ctx.set_stream(stream.cuda_stream)
    src, tgt, _ = synth.eth_pair(seed=1234)
    cfg = capi.default_config()
    cfg.metric, cfg.minimizer, cfg.matching, cfg.n_iterations, cfg.max_distance_sq, cfg.nn_algorithm, cfg.collect_stats = 1, 0, 0, 30, 10.0, 2, 0
    ctx.set_config(cfg)
    for rep in range(4):
        ctx.set_target(tgt.points, tgt.normals, tgt.colors)
        ctx.set_source(src.points, src.normals, src.colors)
        torch.cuda.synchronize()
        if rep == 3:
            lib.icp_gpu_debug_timeline(None, 1)
            lib.icp_gpu_debug_timeline_reduce(None, 1)
            torch.cuda.synchronize()
        ctx.estimate_pose(want_history=False)
        torch.cuda.synchronize()
    tl = np.zeros((2, 2, TL_WARPS, 2), np.uint64)
    tr = np.zeros((512, 2), np.uint64)
    lib.icp_gpu_debug_timeline(tl.ctypes.data_as(C.c_void_p), 0)
    lib.icp_gpu_debug_timeline_reduce(tr.ctypes.data_as(C.c_void_p), 0)
    tl = tl.astype(np.int64); tr = tr.astype(np.int64)
    t0 = tl[0][tl[0][:, :, 0] > 0][:, 0].min()
    out = {"chunks": os.environ.get("ICP_GPU_MATCH_CHUNKS", "default"), "unit": "microseconds from the iteration's first prep warp", "kernels": {}}
    spans = {}
    for k, name in ((0, "prep"), (1, "walk")):
        for c in range(2):
            w = tl[k, c]; w = w[w[:, 0] > 0]
            if len(w) == 0:
                continue
            s = (w[:, 0] - t0) * 1e-3; e = (w[:, 1] - t0) * 1e-3
            life = e - s
            spans[f"{name}{c}"] = (s, e)
            out["kernels"][f"{name}_chunk{c}"] = {
                "warps": int(len(w)), "first_start": round(float(s.min()), 2), "last_start": round(float(s.max()), 2), "end": round(float(e.max()), 2),
                "warp_life_us": {"mean": round(float(life.mean()), 2), "p50": round(float(np.median(life)), 2), "p90": round(float(np.percentile(life, 90)), 2),
                                 "p99": round(float(np.percentile(life, 99)), 2), "max": round(float(life.max()), 2)},
                "time_when_95pct_of_warps_had_ended": round(float(np.percentile(e, 95)), 2),
            }
    b = tr[:511]; b = b[b[:, 0] > 0]
    out["kernels"]["reduce"] = {"blocks": int(len(b)), "first_start": round(float((b[:, 0].min() - t0) * 1e-3), 2),
                                "loops_end": round(float((b[:, 1].max() - t0) * 1e-3), 2), "pose_written": round(float((tr[511, 0] - t0) * 1e-3), 2)}
    # resident search warps per SM over time (all chunks, both kernels), 5 us steps
    end = out["kernels"]["reduce"]["pose_written"]
    grid = np.arange(0.0, end + 5.0, 5.0)
    tot = {}
    for name, (s, e) in spans.items():
        tot[name] = resident(s, e, grid) / 148.0
    out["resident_warps_per_sm_every_5us"] = {name: [round(float(x), 1) for x in v] for name, v in tot.items()}
    print(json.dumps(out))


if __name__ == "__main__":
    main()
