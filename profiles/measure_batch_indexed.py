"""Indexed batched registration (icp_gpu_estimate_pose_batch_indexed) against the same B registrations through a loop of
estimate_pose on one context (set_target + set_source + estimate_pose per pair), alignPairs on three contexts and, where every target
fits its 8192-point stage, estimate_pose_batch; in one run on cuda:0.

Workloads (point-to-plane, identity start, every arm from host arrays):
  - ETH-shaped pairs (synth.eth_pair at reduced sweeps) of ~12.9k (12 sweeps) and ~45k (42 sweeps) points, B = 1, 64 and 512: eight
    generated pairs; every further pair reuses one of their eight targets, and its source is moved by its own seeded rigid motion and
    jittered.  No two sources are the same data, but the targets repeat every eight pairs (each arm still builds one index per pair).
    30 iterations, max distance^2 0.05.
  - eight ETH-shaped pairs cut to 8192 points per cloud (the old batch's limit), 30 iterations.
  - 4096 bunny pairs (seeded perturbations of the source), 20 iterations, max distance^2 0.0003.
Every arm's contexts are created outside the timing and warmed by the untimed first run.  Reported per workload: pairs/s of every
arm, the largest pose difference from the loop, and the build-and-score share: the time of the same call with n_iterations = 0 over
that of the full call.  Times are medians of REPS runs after one warm-up.
Usage: python profiles/measure_batch_indexed.py [out.json]   (default profiles/r6_batch_indexed.json)"""
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from icp_variants_b200 import capi, synth  # noqa: E402
from icp_variants_b200.sequence import alignPairs  # noqa: E402

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
    c.metric, c.minimizer, c.n_iterations, c.max_distance_sq, c.nn_algorithm = 1, 0, n_iterations, max_d2, 0
    return c


def rigid(seed, max_angle, max_trans):
    rng = np.random.default_rng(seed)
    axis = rng.normal(size=3); axis /= np.linalg.norm(axis)
    a = rng.uniform(0.0, max_angle)
    K = np.array([[0, -axis[2], axis[1]], [axis[2], 0, -axis[0]], [-axis[1], axis[0], 0]])
    P = np.eye(4)
    P[:3, :3] = np.eye(3) + np.sin(a) * K + (1 - np.cos(a)) * K @ K
    P[:3, 3] = rng.uniform(-max_trans, max_trans, 3)
    return P


def moved(c, seed, max_angle, max_trans, jitter):
    P = rigid(seed, max_angle, max_trans)
    rng = np.random.default_rng(seed + 1)
    p = (c.points.astype(np.float64) @ P[:3, :3].T + P[:3, 3] + rng.normal(scale=jitter, size=c.points.shape)).astype(np.float32)
    n = (c.normals.astype(np.float64) @ P[:3, :3].T).astype(np.float32)
    return synth.Cloud(p, n, None)


def eth_pairs(n_sweeps, B):
    base = [synth.eth_pair(seed=100 + i, n_sweeps=n_sweeps, n_beams=1077, pair_index=i % 4) for i in range(min(B, 8))]
    pairs = []
    for b in range(B):
        s, t, _ = base[b % len(base)]
        pairs.append((moved(s, 7000 + b, 0.02, 0.02, 0.002) if b >= len(base) else synth.Cloud(s.points, s.normals, None),
                      synth.Cloud(t.points, t.normals, None)))
    return pairs


def loop(ctx, pairs):
    out = []
    for s, t in pairs:
        ctx.set_target(t.points, t.normals); ctx.set_source(s.points, s.normals)
        try:
            out.append(ctx.estimate_pose(None, want_history=False)[0])
        except capi.IcpGpuError as e:
            out.append(e.pose)
    return np.stack(out)


def max_diff(pa, pb):
    r = max(float(np.abs(a[:3, :3].astype(np.float64) - b[:3, :3]).max()) for a, b in zip(pa, pb))
    t = max(float(np.abs(a[:3, 3].astype(np.float64) - b[:3, 3]).max()) for a, b in zip(pa, pb))
    return r, t


def workload(name, pairs, cfg, res, with_batch, loop_reps=REPS):
    B = len(pairs)
    sources, targets = [p[0] for p in pairs], [p[1] for p in pairs]
    ctx = capi.Context(0); ctx.set_config(cfg)
    t_bi, r = median_time(lambda: ctx.estimate_pose_batch_indexed(sources, targets))
    c0 = capi.Config.from_buffer_copy(cfg); c0.n_iterations = 0
    ctx.set_config(c0)
    t_build, _ = median_time(lambda: ctx.estimate_pose_batch_indexed(sources, targets))
    ctx.set_config(cfg)
    lctx = capi.Context(0); lctx.set_config(cfg)
    t_loop, p_loop = median_time(lambda: loop(lctx, pairs), reps=loop_reps)
    ctxs = [capi.Context(0) for _ in range(3)]
    t_al, al = median_time(lambda: alignPairs(ctxs, pairs, cfg), reps=loop_reps)
    dr, dt = max_diff(r["poses"], p_loop)
    w = {"pairs": B, "n_source_mean": float(np.mean([len(s) for s in sources])), "n_target_mean": float(np.mean([len(t) for t in targets])),
         "iterations": cfg.n_iterations, "batch_indexed_ms": t_bi * 1e3, "batch_indexed_pairs_per_s": B / t_bi,
         "build_and_score_ms": t_build * 1e3, "build_and_score_share": t_build / t_bi,
         "loop_estimate_pose_ms": t_loop * 1e3, "loop_pairs_per_s": B / t_loop,
         "alignPairs_3_contexts_ms": t_al * 1e3, "alignPairs_pairs_per_s": B / t_al,
         "speedup_vs_loop": t_loop / t_bi, "speedup_vs_alignPairs": t_al / t_bi,
         "pairs_ok": int((r["status"] == 0).sum()), "max_rot_diff_vs_loop": dr, "max_trans_diff_vs_loop_m": dt,
         "max_rot_diff_vs_alignPairs": max_diff(r["poses"], [a.pose for a in al])[0]}
    if with_batch:
        t_b, rb = median_time(lambda: ctx.estimate_pose_batch(sources, targets))
        w.update(batch_ms=t_b * 1e3, batch_pairs_per_s=B / t_b, speedup_vs_batch=t_b / t_bi, max_rot_diff_vs_batch=max_diff(r["poses"], rb[0])[0])
    for c in ctxs + [ctx, lctx]:
        c.close()
    res[name] = w
    print(name, json.dumps(w), flush=True)


def main():
    out_path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(os.path.dirname(os.path.abspath(__file__)), "r6_batch_indexed.json")
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"], stdout=subprocess.PIPE, text=True)
    res = {}
    report = {"device": q.stdout.strip().split(",")[0], "nvidia_smi_name_power_limit_sm_clock_max_sm_clock": q.stdout.strip(),
              "reps": REPS, "workloads": res}
    eth_cfg = cfg_of(30, 0.05)
    p12 = eth_pairs(12, 512)
    workload("eth12k_B1", p12[:1], eth_cfg, res, False)
    workload("eth12k_B64", p12[:64], eth_cfg, res, False)
    workload("eth12k_B512", p12, eth_cfg, res, False, loop_reps=1)
    p45 = eth_pairs(42, 512)
    workload("eth45k_B64", p45[:64], eth_cfg, res, False)
    workload("eth45k_B512", p45, eth_cfg, res, False, loop_reps=1)
    cut = []
    for s, t in p12[:8]:
        rng = np.random.default_rng(len(cut))
        ks, kt = np.sort(rng.choice(len(s), 8192, replace=False)), np.sort(rng.choice(len(t), 8192, replace=False))
        cut.append((synth.Cloud(s.points[ks], s.normals[ks], None), synth.Cloud(t.points[kt], t.normals[kt], None)))
    workload("eth8192_B8", cut, eth_cfg, res, True)
    bsrc, btgt, _, _ = synth.load_bunny()
    bunny = [(moved(bsrc, 9000 + b, 0.02, 0.002, 0.0), synth.Cloud(btgt.points, btgt.normals, None)) for b in range(4096)]
    workload("bunny_B4096", bunny, cfg_of(20, 0.0003), res, True, loop_reps=1)
    with open(out_path, "w") as f:
        json.dump(report, f, indent=1)


if __name__ == "__main__":
    main()
