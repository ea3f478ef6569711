"""Voxel-grid downsampling on the device (icp_gpu_voxel_downsample[_dev]) against what a user pays without it: the CPU restatement
(tests/voxel_reference.c) on one host core, and the host round trip (download the cloud, filter it on the host, upload the result).
Writes one JSON file.

Workloads: the ~370k-point ETH-shaped scan at 2, 5, 10 and 20 cm; the ~3 M-point scan (1720 x 1744 beams) at 5 cm; batches of 44 and
512 ETH-shaped scans in one call against a loop of single-cloud calls.  Every device timing is the median of --runs calls after
--warmup calls, with CUDA events on the current torch stream around a call that synchronises; L2 is flushed (a 256 MB write) before
every timed call, outside the window.  The card's name, power limit and SM clocks are read in the same run.
Usage: python profiles/measure_voxel.py --out OUT.json"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from icp_variants_b200 import capi, synth  # noqa: E402
sys.path.insert(0, os.path.join(ROOT, "tests"))
import voxel_reference as vref  # noqa: E402


def towards(pts, viewpoint):
    d = np.asarray(viewpoint, np.float64) - pts.astype(np.float64)
    return (d / np.linalg.norm(d, axis=1, keepdims=True)).astype(np.float32)


def scan(n_sweeps, n_beams, pos=(6.0, 4.5, 1.2), seed=7):
    room = synth.make_room(1234)
    return synth.lidar_scan(room, np.array(pos), n_sweeps=n_sweeps, n_beams=n_beams, seed=seed, colors="texture", normals_fn=towards)


def largest_voxel(pts, size):
    inv = np.float32(1.0) / np.float32(size)
    v = np.floor(pts[np.isfinite(pts).all(1)] * inv).astype(np.int64)
    _, counts = np.unique(v, axis=0, return_counts=True)
    return int(counts.max()) if len(counts) else 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--runs", type=int, default=15)
    ap.add_argument("--warmup", type=int, default=3)
    args = ap.parse_args()
    import torch
    dev = torch.device("cuda", 0)
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm,clocks.sm", "--format=csv,noheader"],
                       stdout=subprocess.PIPE, text=True).stdout.strip().splitlines()[0]
    res = {"gpu": q, "runs": args.runs, "warmup": args.warmup, "l2": "flushed (256 MB write) before every timed call, outside the window",
           "timing": "median; device: CUDA events around a call that synchronises; host baselines: one core, perf_counter"}
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    ctx = capi.Context(0)

    def timed(f, runs=args.runs, warmup=args.warmup):
        for _ in range(warmup):
            f()
        ts = []
        for _ in range(runs):
            flush.zero_()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            a.record()
            f()
            b.record()
            b.synchronize()
            ts.append(a.elapsed_time(b))
        return float(np.median(ts)), float(np.min(ts)), float(np.max(ts))

    def host_timed(f, runs=5):
        ts = []
        for _ in range(runs):
            t = time.perf_counter()
            f()
            ts.append((time.perf_counter() - t) * 1e3)
        return float(np.median(ts))

    def single(cloud, size, label):
        xyz, nrm, col = cloud.points, cloud.normals, cloud.colors
        off = np.array([0, len(xyz)], np.int64)
        dx, dn, dc, do = (torch.from_numpy(a).to(dev) for a in (xyz, nrm, col, off))
        host = ctx._voxel_host(xyz, nrm, col, off, size, 2)
        d = ctx.voxel_downsample_dev(dx, do, size, nrm=dn, rgba=dc)
        ref = vref.voxel_downsample(xyz, size, nrm=nrm, rgba=col)
        exact = all(a.tobytes() == b.tobytes() for a, b in zip(host, ref)) and d[0].cpu().numpy().tobytes() == ref[0].tobytes()
        h_med, h_min, h_max = timed(lambda: ctx._voxel_host(xyz, nrm, col, off, size, 2))
        d_med, d_min, d_max = timed(lambda: ctx.voxel_downsample_dev(dx, do, size, nrm=dn, rgba=dc))
        ref_ms = host_timed(lambda: vref.voxel_downsample(xyz, size, nrm=nrm, rgba=col))

        def round_trip():                                     # what a user pays today: download, filter on the host, upload
            hx, hn, hc = dx.cpu().numpy(), dn.cpu().numpy(), dc.cpu().numpy()
            p, n, c, _ = vref.voxel_downsample(hx, size, nrm=hn, rgba=hc)
            torch.from_numpy(p).to(dev); torch.from_numpy(n).to(dev); torch.from_numpy(c).to(dev)
            torch.cuda.synchronize()
        rt_ms = host_timed(round_trip)
        r = {"points": len(xyz), "voxel_m": size, "voxels": int(len(ref[0])), "largest_voxel_points": largest_voxel(xyz, size),
             "bit_exact_vs_reference": bool(exact), "host_form_ms": [h_med, h_min, h_max], "dev_form_ms": [d_med, d_min, d_max],
             "reference_one_core_ms": ref_ms, "host_round_trip_ms": rt_ms,
             "dev_form_vs_round_trip": rt_ms / d_med, "host_form_vs_reference": ref_ms / h_med}
        print(label, json.dumps(r), flush=True)
        return r

    s370 = scan(344, 1077)
    res["scan_370k"] = {f"{int(round(v * 100))}cm": single(s370, v, f"370k {v}") for v in (0.02, 0.05, 0.1, 0.2)}
    s3m = scan(1720, 1744)
    res["scan_3m_5cm"] = single(s3m, 0.05, "3M 0.05")
    del s3m

    def batch(clouds, size, label):
        xyz, nrm, col, off = capi._concat_clouds_rgba(clouds)
        dx, dn, dc, do = (torch.from_numpy(a).to(dev) for a in (xyz, nrm, col, off))
        per = [(torch.from_numpy(c.points).to(dev), torch.from_numpy(np.array([0, len(c.points)], np.int64)).to(dev),
                torch.from_numpy(c.normals).to(dev), torch.from_numpy(c.colors).to(dev)) for c in clouds]
        one = ctx.voxel_downsample_dev(dx, do, size, nrm=dn, rgba=dc)
        oo = one[3].cpu().numpy()
        exact = True
        for b, (px, po, pn, pc) in enumerate(per):
            alone = ctx.voxel_downsample_dev(px, po, size, nrm=pn, rgba=pc)
            exact &= alone[0].cpu().numpy().tobytes() == one[0][oo[b]:oo[b + 1]].cpu().numpy().tobytes()
        b_med, b_min, b_max = timed(lambda: ctx.voxel_downsample_dev(dx, do, size, nrm=dn, rgba=dc), runs=max(5, args.runs // 3))

        def loop():
            for px, po, pn, pc in per:
                ctx.voxel_downsample_dev(px, po, size, nrm=pn, rgba=pc)
        l_med, l_min, l_max = timed(loop, runs=max(5, args.runs // 3), warmup=1)
        h_med, _, _ = timed(lambda: ctx._voxel_host(xyz, nrm, col, off, size, 2), runs=max(5, args.runs // 3))
        r = {"clouds": len(clouds), "points": int(off[-1]), "voxel_m": size, "voxels": int(oo[-1]), "each_equals_alone": bool(exact),
             "batched_dev_ms": [b_med, b_min, b_max], "loop_of_single_dev_ms": [l_med, l_min, l_max], "batched_host_form_ms": h_med,
             "loop_vs_batched": l_med / b_med}
        print(label, json.dumps(r), flush=True)
        return r

    # ETH-shaped scans: 64 distinct ones of ~12.9k points (60 x 215 beams, as the indexed batch's small pairs), repeated in order for
    # B = 512; and the full ~370k-point scan under 44 different rigid motions
    small = [scan(60, 215, pos=(3.0 + 0.2 * (k % 40), 2.0 + 0.15 * (k // 40), 1.2), seed=k) for k in range(64)]
    res["batch_44_small_5cm"] = batch([small[k % 64] for k in range(44)], 0.05, "44 small")
    res["batch_512_small_5cm"] = batch([small[k % 64] for k in range(512)], 0.05, "512 small")
    full = [synth.apply_pose(synth.make_pose(np.array([0.1 * k, 0.05 * k, 0.0]), np.array([0.0, 0.0, 2.0 * k])), s370) for k in range(44)]
    res["batch_44_full_5cm"] = batch(full, 0.05, "44 full")
    res["bunny_4mm"] = single(synth.load_bunny()[0], 0.004, "bunny")
    ctx.close()
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
