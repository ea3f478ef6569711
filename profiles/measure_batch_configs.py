"""Batched registration with one configuration per pair (icp_gpu_estimate_pose_batch_configs) against the same registrations
through a loop of estimate_pose on one context and through sequence.alignPairs on three contexts, in one run on cuda:0.

Workloads:
  - the reference's 24-row bunny matrix ({linear, LM} x {p2p, p2plane, symmetric} x {base, random p = 0.5 mt19937 seed 7,
    distance weights, multires}, 20 iterations, max distance^2 0.0003) x T trials (T = 1, 16, 128) in one call; trial t moves
    the source by its own seeded perturbation, so every path sees identical inputs.  alignPairs takes one configuration per
    call: it runs once per row over that row's T pairs.
  - 4096 LM point-to-plane bunny pairs (own perturbations) in one call; the loop is timed on the first LOOP_CAP pairs and
    reported per pair.
  - the single-configuration entry point's 4096-pair point-to-point workload of profiles/r3_batch.json (icp_gpu_estimate_pose_batch),
    rerun in the same process.
Every path runs the whole registration from host arrays.  Times are medians of REPS runs after a warm-up (the loops at T = 128
and the LM loop: one timed run after the warm-up of the smaller workloads).  Each workload reports the largest pose difference
against the loop.
Usage: python profiles/measure_batch_configs.py [out.json]   (default profiles/r4_batch_configs.json)"""
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from icp_variants_b200 import capi, synth  # noqa: E402
from icp_variants_b200.sequence import alignPairs  # noqa: E402

REPS = 3
LOOP_CAP = 256


def perturbation(seed, max_angle=0.02, max_trans=0.002):
    rng = np.random.default_rng(seed)
    axis = rng.normal(size=3); axis /= np.linalg.norm(axis)
    a = rng.uniform(0.0, max_angle)
    K = np.array([[0, -axis[2], axis[1]], [axis[2], 0, -axis[0]], [-axis[1], axis[0], 0]])
    R = np.eye(3) + np.sin(a) * K + (1 - np.cos(a)) * K @ K
    return R, rng.uniform(-max_trans, max_trans, 3)


def moved(cloud, seed):
    R, t = perturbation(seed)
    p, n = cloud.points.astype(np.float64), cloud.normals.astype(np.float64)
    return synth.Cloud((p @ R.T + t).astype(np.float32), (n @ R.T).astype(np.float32), None)


def median_time(fn, reps=REPS, warm=True):
    if warm:
        fn()
    ts, out = [], None
    for _ in range(reps):
        t0 = time.perf_counter()
        out = fn()
        ts.append(time.perf_counter() - t0)
    return float(np.median(ts)), out


def rot_trans_diff(pa, pb):
    d = np.linalg.norm(pa[:3, :3].astype(np.float64) - pb[:3, :3])
    return float(2.0 * np.arcsin(min(d / (2.0 * np.sqrt(2.0)), 1.0))), float(np.linalg.norm(pa[:3, 3].astype(np.float64) - pb[:3, 3]))


def config(metric, minimizer, **kw):
    c = capi.default_config()
    c.collect_stats = 0
    c.metric, c.minimizer = metric, minimizer
    for k, v in kw.items():
        setattr(c, k, v)
    return c


def matrix():
    variants = [("base", {}), ("random", dict(selection=1, proba=0.5, seed=7, selection_rng=0)), ("distance_weights", dict(weighting=1)),
                ("multires", dict(multires=1))]
    return [(f"{'lm' if mi else 'linear'}_{('p2p', 'p2plane', 'symmetric')[me]}_{name}", config(me, mi, **kw))
            for mi in (0, 1) for me in (0, 1, 2) for name, kw in variants]


def loop(ctx, cfgs, ci, srcs, tgts):
    out = []
    for k, s, t in zip(ci, srcs, tgts):
        ctx.set_config(cfgs[k])
        ctx.set_target(t.points, t.normals, t.colors)
        ctx.set_source(s.points, s.normals, s.colors)
        try:
            out.append(ctx.estimate_pose(want_history=False)[0])
        except capi.IcpGpuError as e:
            out.append(e.pose)
    return out


def main():
    out_path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(os.path.dirname(os.path.abspath(__file__)), "r4_batch_configs.json")
    torch.cuda.set_device(0)
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"], stdout=subprocess.PIPE, text=True)
    ctxs = [capi.Context(0) for _ in range(3)]
    ctx = ctxs[0]
    res = {"device": torch.cuda.get_device_name(0), "nvidia_smi_name_power_limit_sm_clock_max_sm_clock": q.stdout.strip(), "reps": REPS,
           "workloads": {}}
    src, tgt, _, _ = synth.load_bunny()
    rows = matrix()
    cfgs = [c for _, c in rows]
    for T in (1, 16, 128):
        srcs = [moved(src, 3000 + t) for t in range(T) for _ in rows]
        tgts = [tgt] * len(srcs)
        ci = np.tile(np.arange(len(rows), dtype=np.int32), T)
        B = len(ci)
        t_batch, (poses, n_it, status) = median_time(lambda: ctx.estimate_pose_batch_configs(cfgs, ci, srcs, tgts))
        big = T >= 128
        t_loop, lposes = median_time(lambda: loop(ctx, cfgs, ci, srcs, tgts), reps=1 if big else REPS, warm=not big)

        def per_row():
            for k, (_, c) in enumerate(rows):
                alignPairs(ctxs, [(srcs[b], tgts[b]) for b in range(k, B, len(rows))], c)
        t_ap, _ = median_time(per_row, reps=1 if big else REPS, warm=not big)
        diffs = [rot_trans_diff(poses[b], lposes[b]) for b in range(B)]
        r = {"pairs": B, "trials": T, "pairs_ok": int((status == capi.OK).sum()), "iterations_mean": float(np.mean(n_it)),
             "batch_ms": t_batch * 1e3, "batch_pairs_per_s": B / t_batch,
             "loop_estimate_pose_ms": t_loop * 1e3, "loop_pairs_per_s": B / t_loop,
             "alignPairs_3_contexts_per_row_ms": t_ap * 1e3, "alignPairs_pairs_per_s": B / t_ap,
             "batch_speedup_vs_loop": t_loop / t_batch, "batch_speedup_vs_alignPairs": t_ap / t_batch,
             "max_rot_diff_vs_loop_rad": max(d[0] for d in diffs), "max_trans_diff_vs_loop_m": max(d[1] for d in diffs)}
        # per row: the batch's share is not separable (one call), the loop's is
        print(f"matrix x {T}", json.dumps(r), flush=True)
        res["workloads"][f"bunny_matrix24_x{T}"] = r

    lm = config(1, 1)
    B = 4096
    srcs = [moved(src, 1000 + b) for b in range(B)]
    tgts = [tgt] * B
    ci = np.zeros(B, np.int32)
    t_batch, (poses, n_it, status) = median_time(lambda: ctx.estimate_pose_batch_configs([lm], ci, srcs, tgts))
    t_loop, lposes = median_time(lambda: loop(ctx, [lm], ci[:LOOP_CAP], srcs[:LOOP_CAP], tgts[:LOOP_CAP]), reps=1)
    diffs = [rot_trans_diff(poses[b], lposes[b]) for b in range(LOOP_CAP)]
    r = {"pairs": B, "pairs_ok": int((status == capi.OK).sum()), "iterations_mean": float(np.mean(n_it)),
         "batch_ms": t_batch * 1e3, "batch_pairs_per_s": B / t_batch,
         "loop_pairs_timed": LOOP_CAP, "loop_ms_per_pair": t_loop * 1e3 / LOOP_CAP, "loop_pairs_per_s": LOOP_CAP / t_loop,
         "batch_speedup_vs_loop": (B / t_batch) / (LOOP_CAP / t_loop),
         "max_rot_diff_vs_loop_rad": max(d[0] for d in diffs), "max_trans_diff_vs_loop_m": max(d[1] for d in diffs)}
    print("lm p2plane 4096", json.dumps(r), flush=True)
    res["workloads"]["bunny_lm_p2plane_20it_B4096"] = r

    old = config(0, 0)                                             # r3_batch.json's bunny_p2p_20it_B4096
    ctx.set_config(old)
    t_old, (poses_old, _, _) = median_time(lambda: ctx.estimate_pose_batch(srcs, tgts))
    t_new, (poses_new, _, _) = median_time(lambda: ctx.estimate_pose_batch_configs([old], ci, srcs, tgts))
    r = {"pairs": B, "estimate_pose_batch_ms": t_old * 1e3, "estimate_pose_batch_pairs_per_s": B / t_old,
         "estimate_pose_batch_configs_ms": t_new * 1e3, "estimate_pose_batch_configs_pairs_per_s": B / t_new,
         "identical_poses": bool(np.array_equal(poses_old, poses_new)), "r3_batch_json_pairs_per_s": 24500}
    print("old entry p2p 4096", json.dumps(r), flush=True)
    res["workloads"]["bunny_p2p_20it_B4096_old_entry"] = r
    os.makedirs(os.path.dirname(out_path) or ".", exist_ok=True)
    with open(out_path, "w") as f:
        json.dump(res, f, indent=1)
    for c in ctxs:
        c.close()


if __name__ == "__main__":
    main()
