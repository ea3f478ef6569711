"""Batched registration of many small pairs (icp_gpu_estimate_pose_batch, one thread block per pair) against the same pairs
through (a) a loop of estimate_pose on one context and (b) sequence.alignPairs on three contexts, in one run on cuda:0.

Workloads: the bunny pair x B = 1, 148, 1024, 4096 (each copy's source moved by its own seeded perturbation, identity start
pose, so all three paths see identical inputs); a 24-pair mix of bunny trials (source strides 1 / 2 / 3, own perturbations);
8 ETH-shaped scan pairs cut to their first 8192 points.  Every path runs the whole registration from host arrays (uploads,
for the single-pair paths also the index build); the batch is also timed with CUDA events on the device-resident form
(estimate_pose_batch_dev on the torch stream).  Distance evaluations: every query of every executed iteration scans the
pair's whole target; rate against the measured FP32 FMUL+FADD rate (icp_gpu_measure_fp32_peak mode 1), 8 flop per
evaluation (D1: 3 sub, 3 mul, 2 add).  Times are medians of `REPS` runs after a warm-up.
Usage: python profiles/measure_batch.py [out.json]   (default profiles/r3_batch.json)"""
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


def perturbation(seed, max_angle=0.02, max_trans=0.002):
    rng = np.random.default_rng(seed)
    axis = rng.normal(size=3); axis /= np.linalg.norm(axis)
    a = rng.uniform(0.0, max_angle)
    K = np.array([[0, -axis[2], axis[1]], [axis[2], 0, -axis[0]], [-axis[1], axis[0], 0]])
    R = np.eye(3) + np.sin(a) * K + (1 - np.cos(a)) * K @ K
    return R, rng.uniform(-max_trans, max_trans, 3)


def moved(cloud, seed, stride=1, **kw):
    R, t = perturbation(seed, **kw)
    p, n = cloud.points[::stride].astype(np.float64), cloud.normals[::stride].astype(np.float64)
    return synth.Cloud((p @ R.T + t).astype(np.float32), (n @ R.T).astype(np.float32), None)


def median_time(fn):
    fn()                                           # warm-up: allocations, graph capture
    ts = []
    for _ in range(REPS):
        t0 = time.perf_counter()
        out = fn()
        ts.append(time.perf_counter() - t0)
    return float(np.median(ts)), out


def rot_trans_diff(pa, pb):
    d = np.linalg.norm(pa[:3, :3].astype(np.float64) - pb[:3, :3])
    return float(2.0 * np.arcsin(min(d / (2.0 * np.sqrt(2.0)), 1.0))), float(np.linalg.norm(pa[:3, 3].astype(np.float64) - pb[:3, 3]))


def run(name, pairs, cfg, ctxs, peak_tflops, loops=True):
    srcs, tgts = [p[0] for p in pairs], [p[1] for p in pairs]
    B = len(pairs)
    ctx = ctxs[0]
    ctx.set_config(cfg)
    t_batch, (poses, n_it, status) = median_time(lambda: ctx.estimate_pose_batch(srcs, tgts))
    # device-resident form on the torch stream, CUDA events
    dev = torch.device("cuda", 0)
    sp, sn, so = capi._concat_clouds(srcs)
    tp, tn, to = capi._concat_clouds(tgts)
    g = [torch.from_numpy(a).to(dev) for a in (sp, so, tp, to, sn, tn)]
    stream = torch.cuda.current_stream()
    ctx.set_stream(stream.cuda_stream)
    ev = []
    for i in range(REPS + 1):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        dposes, _, _ = ctx.estimate_pose_batch_dev(*g)
        e1.record(stream)
        e1.synchronize()
        if i > 0:
            ev.append(e0.elapsed_time(e1))
    ctx.set_stream(None)
    t_dev = float(np.median(ev)) * 1e-3
    assert np.array_equal(dposes.cpu().numpy(), poses), "device form differs from the host form"
    executed = n_it + (status != capi.OK)
    evals = float(sum(int(e) * len(s) * len(t) for e, s, t in zip(executed, srcs, tgts)))
    r = {"pairs": B, "source_points": int(sum(len(s) for s in srcs)), "target_points_max": int(max(len(t) for t in tgts)),
         "iterations_mean": float(np.mean(n_it)), "pairs_ok": int((status == capi.OK).sum()),
         "batch_host_ms": t_batch * 1e3, "batch_host_pairs_per_s": B / t_batch,
         "batch_device_resident_event_ms": t_dev * 1e3, "batch_device_resident_pairs_per_s": B / t_dev,
         "distance_evals": evals, "distance_evals_per_s": evals / t_dev,
         "fp32_share_of_measured_fmul_fadd_rate": evals * 8 / t_dev / (peak_tflops * 1e12)}
    if loops:
        def loop():
            out = []
            for s, t in zip(srcs, tgts):
                ctx.set_target(t.points, t.normals, t.colors)
                ctx.set_source(s.points, s.normals, s.colors)
                try:
                    out.append(ctx.estimate_pose(want_history=False)[0])
                except capi.IcpGpuError as e:
                    out.append(e.pose)
            return out
        t_loop, lposes = median_time(loop)
        t_ap, _ = median_time(lambda: alignPairs(ctxs, pairs, cfg))
        diffs = [rot_trans_diff(poses[b], lposes[b]) for b in range(B)]
        r.update({"loop_estimate_pose_ms": t_loop * 1e3, "loop_pairs_per_s": B / t_loop,
                  "alignPairs_3_contexts_ms": t_ap * 1e3, "alignPairs_pairs_per_s": B / t_ap,
                  "batch_speedup_vs_loop": t_loop / t_batch, "batch_speedup_vs_alignPairs": t_ap / t_batch,
                  "max_rot_diff_vs_loop_rad": max(d[0] for d in diffs), "max_trans_diff_vs_loop_m": max(d[1] for d in diffs)})
    print(name, json.dumps(r), flush=True)
    return r


def main():
    out_path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(os.path.dirname(os.path.abspath(__file__)), "r3_batch.json")
    torch.cuda.set_device(0)
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], stdout=subprocess.PIPE, text=True)
    ctxs = [capi.Context(0) for _ in range(3)]
    peak = ctxs[0].measure_fp32_peak(1)
    res = {"device": torch.cuda.get_device_name(0), "nvidia_smi_name_power_limit_max_sm_clock": q.stdout.strip(),
           "fp32_fmul_fadd_tflops_measured": peak, "reps": REPS, "workloads": {}}
    src, tgt, _, _ = synth.load_bunny()
    bunny = capi.default_config(); bunny.collect_stats = 0               # C1: p2p, 20 iterations, max_distance_sq 0.0003
    for B in (1, 148, 1024, 4096):
        pairs = [(moved(src, 1000 + b), tgt) for b in range(B)]
        res["workloads"][f"bunny_p2p_20it_B{B}"] = run(f"bunny B={B}", pairs, bunny, ctxs, peak)
    mix = capi.default_config(); mix.collect_stats = 0; mix.metric = 1
    pairs = [(moved(src, 2000 + b, stride=1 + b % 3), tgt) for b in range(24)]
    res["workloads"]["bunny_mix24_p2plane_20it"] = run("bunny mix 24", pairs, mix, ctxs, peak)
    eth = capi.default_config(); eth.collect_stats = 0; eth.metric = 1; eth.n_iterations = 30; eth.max_distance_sq = 0.1
    pairs = []
    for k in range(8):
        s, t, _ = synth.eth_pair(seed=1234, n_sweeps=56, n_beams=160, pair_index=k)
        n = capi.BATCH_MAX_TARGET                                        # the first 8192 points of each scan
        pairs.append((synth.Cloud(s.points[:n].copy(), s.normals[:n].copy(), None), synth.Cloud(t.points[:n].copy(), t.normals[:n].copy(), None)))
    res["workloads"]["eth8k_x8_p2plane_30it"] = run("eth 8k x 8", pairs, eth, ctxs, peak)
    os.makedirs(os.path.dirname(out_path) or ".", exist_ok=True)
    with open(out_path, "w") as f:
        json.dump(res, f, indent=1)
    for c in ctxs:
        c.close()


if __name__ == "__main__":
    main()
