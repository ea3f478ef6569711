"""Multi-start registration (icp_gpu_estimate_pose_multistart) against the same K registrations through a loop of estimate_pose on
one context (the index built once) and through estimate_pose_async on three contexts, in one run on cuda:0.

Workloads:
  - the bench's 370k-point ETH-shaped pair (synth.eth_pair(seed=1234), point-to-plane, 30 iterations, max distance^2 10): the target
    indexed once, the source its 1-in-32 subsample (K = 1, 8, 24, 148, 1024) or the whole source (K = 1, 8, 24, 148); start k is
    the pose of yaw -30 + 60 k / K degrees and translation 0.02 (k mod 5) m.
  - the bunny, K = 4096 seeded perturbations (point-to-plane, 20 iterations): the multi-start call against estimate_pose_batch
    with K copies of the target.
  - the n_iterations = 0 scorer on the subsampled ETH pair (poses verified per second).
Every path takes host arrays and returns host arrays.  Times are medians of REPS runs after one warm-up.  Each workload reports
the largest pose difference against the loop.
Usage: python profiles/measure_multistart.py [out.json]   (default profiles/r5_multistart.json)"""
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from icp_variants_b200 import capi, synth  # noqa: E402

REPS = 3


def median_time(fn, reps=REPS):
    fn()
    ts, out = [], None
    for _ in range(reps):
        t0 = time.perf_counter()
        out = fn()
        ts.append(time.perf_counter() - t0)
    return float(np.median(ts)), out


def cfg_of(n_iterations, max_d2):
    c = capi.default_config()
    c.metric, c.minimizer, c.n_iterations, c.max_distance_sq, c.nn_algorithm = 1, 0, n_iterations, max_d2, 2
    return c


def starts_eth(K):
    return np.stack([synth.make_pose(np.array([0.02 * (k % 5), 0.0, 0.0]), (0.0, 0.0, -30.0 + 60.0 * k / K)).astype(np.float32) for k in range(K)])


def perturbation(seed, max_angle=0.02, max_trans=0.002):
    rng = np.random.default_rng(seed)
    axis = rng.normal(size=3); axis /= np.linalg.norm(axis)
    a = rng.uniform(0.0, max_angle)
    K = np.array([[0, -axis[2], axis[1]], [axis[2], 0, -axis[0]], [-axis[1], axis[0], 0]])
    P = np.eye(4)
    P[:3, :3] = np.eye(3) + np.sin(a) * K + (1 - np.cos(a)) * K @ K
    P[:3, 3] = rng.uniform(-max_trans, max_trans, 3)
    return P.astype(np.float32)


def max_diff(pa, pb):
    r = max(float(np.abs(a[:3, :3].astype(np.float64) - b[:3, :3]).max()) for a, b in zip(pa, pb))
    t = max(float(np.abs(a[:3, 3].astype(np.float64) - b[:3, 3]).max()) for a, b in zip(pa, pb))
    return r, t


def loop(ctx, starts):
    out = []
    for s in starts:
        try:
            out.append(ctx.estimate_pose(s, want_history=False)[0])
        except capi.IcpGpuError as e:
            out.append(e.pose)
    return np.stack(out)


def async3(ctxs, starts):
    out = [None] * len(starts)
    for b in range(0, len(starts), len(ctxs)):
        for j, c in enumerate(ctxs):
            if b + j < len(starts):
                c.estimate_pose_async(starts[b + j])
        for j, c in enumerate(ctxs):
            if b + j < len(starts):
                try:
                    out[b + j] = c.estimate_pose_finish()[0]
                except capi.IcpGpuError as e:
                    out[b + j] = np.full((4, 4), np.nan, np.float32)
    return np.stack(out)


def eth_workload(src, tgt, cfg, Ks, name, res):
    ctxs = []
    for _ in range(3):
        c = capi.Context(0); c.set_config(cfg); c.set_target(tgt.points, tgt.normals); c.set_source(src.points, src.normals)
        ctxs.append(c)
    ctx = ctxs[0]
    for K in Ks:
        starts = starts_eth(K)
        t_ms, r = median_time(lambda: ctx.estimate_pose_multistart(starts))
        t_loop, p_loop = median_time(lambda: loop(ctx, starts))
        t_async, _ = median_time(lambda: async3(ctxs, starts))
        dr, dt = max_diff(r["poses"], p_loop)
        res[f"{name}_K{K}"] = {"n_source": len(src.points), "n_target": len(tgt.points), "starts": K, "iterations": cfg.n_iterations,
                               "multistart_ms": t_ms * 1e3, "multistart_starts_per_s": K / t_ms,
                               "loop_estimate_pose_ms": t_loop * 1e3, "loop_starts_per_s": K / t_loop,
                               "async_3_contexts_ms": t_async * 1e3, "async_starts_per_s": K / t_async,
                               "speedup_vs_loop": t_loop / t_ms, "speedup_vs_async": t_async / t_ms,
                               "starts_ok": int((r["status"] == 0).sum()), "best": r["best"], "best_inliers": int(r["inliers"][r["best"]]),
                               "max_rot_diff_vs_loop": dr, "max_trans_diff_vs_loop_m": dt}
        print(name, K, json.dumps(res[f"{name}_K{K}"]), flush=True)
    for c in ctxs:
        c.close()


def main():
    out_path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(os.path.dirname(os.path.abspath(__file__)), "r5_multistart.json")
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"], stdout=subprocess.PIPE, text=True)
    res = {}
    report = {"device": q.stdout.strip().split(",")[0], "nvidia_smi_name_power_limit_sm_clock_max_sm_clock": q.stdout.strip(),
              "reps": REPS, "workloads": res}
    src, tgt, _ = synth.eth_pair(seed=1234)
    sub = synth.Cloud(src.points[::32].copy(), src.normals[::32].copy(), None)
    cfg = cfg_of(30, 10.0)
    eth_workload(sub, tgt, cfg, (1, 8, 24, 148, 1024), "eth_sub32", res)
    eth_workload(src, tgt, cfg, (1, 8, 24, 148), "eth_full", res)

    # the scorer: n_iterations = 0
    ctx = capi.Context(0); ctx.set_config(cfg_of(0, 10.0)); ctx.set_target(tgt.points, tgt.normals); ctx.set_source(sub.points, sub.normals)
    starts = starts_eth(1024)
    t, _ = median_time(lambda: ctx.estimate_pose_multistart(starts))
    res["eth_sub32_scorer_K1024"] = {"n_source": len(sub.points), "poses": 1024, "ms": t * 1e3, "poses_per_s": 1024 / t}
    print(json.dumps(res["eth_sub32_scorer_K1024"]), flush=True)
    ctx.close()

    # bunny, K = 4096: multi-start against the batch with K target copies
    bsrc, btgt, _, _ = synth.load_bunny()
    bcfg = cfg_of(20, 0.0003)
    ctx = capi.Context(0); ctx.set_config(bcfg); ctx.set_target(btgt.points, btgt.normals); ctx.set_source(bsrc.points, bsrc.normals)
    K = 4096
    starts = np.stack([perturbation(s) for s in range(K)])
    t_ms, r = median_time(lambda: ctx.estimate_pose_multistart(starts))
    t_b, rb = median_time(lambda: ctx.estimate_pose_batch([bsrc] * K, [btgt] * K, starts))
    t_loop, p_loop = median_time(lambda: loop(ctx, starts[:256]), reps=1)
    dr, dt = max_diff(r["poses"][:256], p_loop)
    res["bunny_K4096"] = {"n_source": len(bsrc.points), "n_target": len(btgt.points), "starts": K, "multistart_ms": t_ms * 1e3,
                          "multistart_starts_per_s": K / t_ms, "batch_ms": t_b * 1e3, "batch_starts_per_s": K / t_b,
                          "loop_starts_per_s_first256": 256 / t_loop, "speedup_vs_batch": t_b / t_ms,
                          "max_rot_diff_vs_loop_first256": dr, "max_trans_diff_vs_loop_first256_m": dt,
                          "max_rot_diff_vs_batch": max_diff(r["poses"], rb[0])[0]}
    print(json.dumps(res["bunny_K4096"]), flush=True)
    with open(out_path, "w") as f:
        json.dump(report, f, indent=1)


if __name__ == "__main__":
    main()
