#!/usr/bin/env python
"""bench.py -- the registration hot path on B200, measured.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]

One STEP = one complete ICP registration of the workload BASELINE.json quotes its metric on
(configs[1]): an ETH-Apartment-shaped synthetic scan pair (344 sweeps x 1077 beams, ~370k points
per scan), k-NN matching, point-to-plane linear ICP, 30 iterations, select-all, constant weights,
normal-angle rejection on -- including the index build (the reference does buildIndex inside
estimatePose, ICPOptimizer.h:532-535).

  value    registrations/s with the raw clouds already resident in HBM (device pointers in, pose out)
  e2e      the same registration through the host-pointer C ABI call a reference user would make
           (icp_gpu_set_target / set_source / estimate_pose with host arrays): the H2D copy of both
           clouds and the D2H read of the pose are inside the timed region
  roofline the dominant kernel (the warp-per-query tree walk of the k-NN search), CUDA-event timed per launch;
           roofline_fp32 relates its distance evaluations to the device's FP32 throughput MEASURED in the same run
  cpu_baseline  (N = 1) the reference's own LinearICPOptimizer::estimatePose (oracle/_ref: the reference headers compiled in
           place against the stand-ins of oracle/ref_shim) on the same pair: one FULL 30-iteration registration on all host
           threads, a bounded 1-thread sample, and the FLANN-like approximate matcher (cv2.flann_Index, 1 tree, 16 checks)
           with its match rate against the exact search
  pair_queue_44  config 5a: a 44-pair ETH-shaped sequence, one queue per GPU, no collective on the data path: the ranks draw pair
           indices from a shared ticket counter (--static-deal: round-robin), host arrays in, poses out -- pairs/s over all
           ranks and the ceiling 44 / ceil(44 / N)
  sharded_3m     config 5b: ONE 3 M-point pair sharded by source points over the ranks, the per-iteration all-reduce of the 28-double
           row fused into the reduction kernel over NVLink peer memory (icp_gpu_peer_*), next to an ncclAllReduce on the stream

N > 1 (torchrun): `value` = independent pairs, one per rank per step -> weak scaling; time = max over ranks.

--impl reference: times the reference's own code path -- LinearICPOptimizer::estimatePose from
/root/reference/icp-variants/ICPOptimizer.h, compiled in place into oracle/_ref/libicp_ref.so -- on the box's host
cores: every step is one FULL 30-iteration registration of the same pair (no extrapolation).  Eigen, FLANN, Ceres and PCL
are neither vendored nor installed, so that build uses the stand-ins of oracle/ref_shim: the matcher is an EXACT kd-tree
(OpenMP over the queries, all host threads) instead of FLANN's approximate one, the 4M x 6 least squares a Gram-matrix
SVD; every other line (transforms with a 3x3 inverse per normal, weighting, rejection, gather, system assembly, pose
composition) is the reference's own, single-threaded as in the reference.  Without the library the arm falls back to the
oracle port (kind "port").
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

N_ITER = 30
WORKLOAD = "eth_apartment_shaped_pair_344x1077_knn_point_to_plane_linear_30it"
N_SEQUENCE_PAIRS = 44
L2_NOTE = "GPU arm: flushed between timed steps (256 MB write); CPU arm: not applicable"


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return float(d.get("hbm_gbs", 6650.0)), "measured"
    return 6650.0, "fallback"


def ncu_traffic(kernel_substr):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of a kernel, from the newest committed ncu --set full capture
    (profiles/r2_ncu_traffic.json, else round 1's); None when the summary is absent."""
    for name in ("r2_ncu_traffic.json", "r1_ncu_traffic.json"):
        try:
            with open(os.path.join(ROOT, "profiles", name)) as f:
                k = json.load(f)["kernels"]
            for kn, v in k.items():
                if kernel_substr in kn:
                    return v["dram_bytes_read"] + v["dram_bytes_write"]
        except Exception:   # noqa: BLE001
            continue
    return None


def _load_pair_cache(cache):
    """A cached pair, or None when the file is absent or unreadable (a run killed while writing it)."""
    from icp_variants_b200 import synth
    if not os.path.exists(cache):
        return None
    try:
        z = np.load(cache)
        return (synth.Cloud(z["sp"], z["sn"], z["sc"]), synth.Cloud(z["tp"], z["tn"], z["tc"]))
    except Exception:   # noqa: BLE001
        return None


def _save_pair_cache(cache, src, tgt):
    """Written under a private name and renamed: other ranks read these files (pair_queue_44's dynamic deal)."""
    tmp = f"{cache}.{os.getpid()}.tmp.npz"
    try:
        np.savez(tmp, sp=src.points, sn=src.normals, sc=src.colors, tp=tgt.points, tn=tgt.normals, tc=tgt.colors)
        os.replace(tmp, cache)
    except OSError:
        try:
            os.remove(tmp)
        except OSError:
            pass


def make_pair(pair_index=0, n_sweeps=344, n_beams=1077):
    """Synthetic ETH-shaped pair; cached in the temporary directory because k=5 PCA normals of 370k points take seconds."""
    from icp_variants_b200 import synth
    cache = os.path.join(tempfile.gettempdir(), f"icp_b200_pair_{n_sweeps}x{n_beams}_{pair_index}.npz")
    hit = _load_pair_cache(cache)
    if hit is not None:
        return hit
    src, tgt, _ = synth.eth_pair(seed=1234, n_sweeps=n_sweeps, n_beams=n_beams, pair_index=pair_index)
    _save_pair_cache(cache, src, tgt)
    return src, tgt


def device_normals_fn(ctx):
    """k = 5 PCA normals towards the sensor on the device (icp_gpu_target_normals = PointCloud.h:41-76): input preparation of
    the big synthetic workloads only (never inside a timed region)."""
    def f(points, viewpoint):
        ctx.set_target(points, None, None)
        return ctx.target_normals(5, viewpoint, n=len(points))
    return f


def make_pair_device_normals(ctx, pair_index, n_sweeps, n_beams):
    from icp_variants_b200 import synth
    cache = os.path.join(tempfile.gettempdir(), f"icp_b200_pairdn_{n_sweeps}x{n_beams}_{pair_index}.npz")
    hit = _load_pair_cache(cache)
    if hit is not None:
        return hit
    src, tgt, _ = synth.eth_pair(seed=1234, n_sweeps=n_sweeps, n_beams=n_beams, pair_index=pair_index, normals_fn=device_normals_fn(ctx))
    _save_pair_cache(cache, src, tgt)
    return src, tgt


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i", str(self.index), "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
            except (ValueError, IndexError):
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def dump_outputs(out_dir, arrays):
    """--dump-outputs: one DIR/<name>.npy (float32) per array, so that two builds can be compared output for output on the
    same seeded inputs."""
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), np.asarray(a, dtype=np.float32))


def workload_config(ns, nt, max_d2):
    """The workload both arms run (BASELINE.json configs[1]); identical in both arms' lines."""
    return {"workload": WORKLOAD, "n_source": ns, "n_target": nt, "iterations": N_ITER, "max_distance_sq": max_d2,
            "pairs_per_gpu_per_step": 1, "includes_index_build": True, "l2": L2_NOTE}


# ----------------------------------------------------------------------------- CPU arms
def host_threads():
    return os.cpu_count() or 1


def ref_registration(src, tgt, max_d2, iters, threads):
    """The reference's own LinearICPOptimizer::estimatePose (oracle/_ref) for `iters` iterations on `threads` matcher threads.
    Returns (seconds, pose), or None when the library is unavailable."""
    try:
        from oracle import ref
        if ref.build() is None:
            return None
        ref.set_num_threads(threads)
        t0 = time.perf_counter()
        n, pose, _ = ref.estimate_pose(0, 1, src.points, src.normals, src.colors, tgt.points, tgt.normals, tgt.colors,
                                       src.points[:4], tgt.points[:4], n_iterations=iters, max_distance_sq=max_d2)
        dt = time.perf_counter() - t0
        return (dt, pose) if n == iters else None
    except Exception as e:   # noqa: BLE001 -- the baseline must never take the bench down
        print(f"bench: reference library unavailable ({e}); using the oracle port", file=sys.stderr)
        return None


def port_registration(src, tgt, max_d2, iters, threads):
    """The oracle's whole registration loop (kind "port") -- only when oracle/_ref is absent."""
    from oracle import oracle as orc
    orc.build()
    orc.set_num_threads(threads)
    cfg = orc.Config(metric=1, minimizer=0, max_distance_sq=max_d2, n_iterations=iters)
    t0 = time.perf_counter()
    _, pose, _, _ = orc.estimate_pose(cfg, src.points, src.normals, src.colors, tgt.points, tgt.normals, tgt.colors)
    return time.perf_counter() - t0, pose


def cpu_registration(src, tgt, max_d2, iters, threads):
    """(seconds, kind, pose) of one CPU registration of `iters` iterations."""
    r = ref_registration(src, tgt, max_d2, iters, threads)
    if r is not None:
        return r[0], "reference", r[1]
    dt, pose = port_registration(src, tgt, max_d2, iters, threads)
    return dt, "port", pose


def cpu_baseline_block(src, tgt, max_d2):
    """cpu_baseline of the GPU arm's line: one full registration on all host threads (the value), a bounded 1-thread sample, and
    the FLANN-like approximate matcher with its match rate."""
    cores = host_threads()
    dt, kind, _ = cpu_registration(src, tgt, max_d2, N_ITER, cores)
    out = {"value": 1.0 / dt, "unit": "reg/s", "cores": cores, "kind": kind, "seconds": dt,
           "sample": f"one full {N_ITER}-iteration registration of the same {len(src)}-point pair (index build included), exact kd-tree matcher on "
                     f"{cores} OpenMP threads, the rest of the loop single-threaded as in the reference"}
    # the reference is single-threaded apart from Ceres (no OpenMP flag, CMakeLists.txt:50-63): 1-thread figure from a bounded sample
    t1, _, _ = cpu_registration(src, tgt, max_d2, 1, 1)
    t2, _, _ = cpu_registration(src, tgt, max_d2, 2, 1)
    one = t1 + (N_ITER - 1) * max(t2 - t1, 0.0)
    out["one_core"] = {"value": 1.0 / one, "unit": "reg/s", "cores": 1, "seconds_estimated": one,
                       "sample": f"bounded: a 1-iteration ({t1:.2f} s) and a 2-iteration ({t2:.2f} s) run on one thread, extended to {N_ITER} iterations "
                                 "(index build counted once)"}
    try:
        from oracle import flann_like
        if flann_like.available():
            r = flann_like.register_p2plane(src, tgt, max_d2, 3)
            per_it = statistics.mean(r["seconds_per_iteration"])
            est = r["seconds_build"] + N_ITER * per_it
            out["flann_like"] = {"value": 1.0 / est, "unit": "reg/s", "cores": 1, "seconds_estimated": est, "seconds_per_iteration": per_it,
                                 "match_rate_vs_exact": r["match_rate"], "matched_fraction_exact": r["matched_fraction"],
                                 "sample": "bounded: 3 iterations of the same pair with cv2.flann_Index(KDTREE, trees=1), checks=16 -- the stand-in for "
                                           "FLANN 1.8.4 KDTreeIndexParams(1) / SearchParams(16) (NearestNeighbor.h:136,172-174) -- extended to 30 iterations"}
    except Exception as e:   # noqa: BLE001
        out["flann_like"] = {"unavailable": str(e)}
    return out


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    src, tgt = make_pair(0, args.sweeps, args.beams)
    cores = host_threads()
    os.environ["OMP_NUM_THREADS"] = str(cores)          # torchrun exports 1; the baseline may use every host core
    kind = "port"
    for _ in range(args.warmup):
        _, kind, _ = cpu_registration(src, tgt, args.max_dist2, N_ITER, cores)
    times = []
    for _ in range(args.steps):
        dt, kind, pose = cpu_registration(src, tgt, args.max_dist2, N_ITER, cores)
        times.append(dt)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"pose": pose})
    per_reg = statistics.mean(times)
    value = 1.0 / per_reg
    sample = (f"every step = one full {N_ITER}-iteration registration of the same {len(src)}-point pair (index build included); exact kd-tree "
              f"matcher on {cores} OpenMP threads, the rest of the loop single-threaded as in the reference")
    line = {"impl": "reference", "metric": "icp_registrations_per_s", "value": value, "unit": "reg/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": per_reg * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": workload_config(len(src), len(tgt), args.max_dist2),
            "mcorr_per_s": len(src) * N_ITER / per_reg / 1e6,
            "cpu_baseline": {"value": value, "unit": "reg/s", "cores": cores, "kind": kind, "sample": sample},
            "e2e": {"value": value, "unit": "reg/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "note": ("reference's own estimatePose compiled in place (oracle/_ref); Eigen/FLANN absent: exact kd-tree matcher on all host threads "
                     "instead of FLANN's approximate search, Gram-matrix SVD; the rest of the loop is the reference's single-threaded code"
                     if kind == "reference" else "oracle/_ref absent: oracle port, exact kd-tree instead of FLANN's approximate search")}
    print(json.dumps(line))
    return 0


# ----------------------------------------------------------------------------- multi-GPU workloads (config 5)
def pair_queue_block(torch, dist, capi, ctx, stream, world, rank, dev, args):
    """Config 5a: the 44 pairs of an ETH-Apartment-shaped sequence dealt round-robin (parallel.shard_pairs) to the ranks; every
    rank runs its queue through sequence.alignPairs (host arrays in, poses out, three contexts per GPU so that the upload and the
    loops of different pairs overlap).  No collective on the data path; time = CUDA events around the queue, max over ranks."""
    from icp_variants_b200 import parallel, sequence, synth
    # the ticket counter lives in the process group's store (same torch on every rank: the same answer everywhere)
    dynamic = world > 1 and not args.static_deal and hasattr(dist.distributed_c10d, "_get_default_store")
    mine = parallel.shard_pairs(N_SEQUENCE_PAIRS, world, rank)
    t0 = time.perf_counter()
    pairs = {k: make_pair_device_normals(ctx, k, args.sweeps, args.beams) for k in mine}     # (also fills the pair cache)
    if dynamic:
        # every rank must be able to read every pair: the ranks generated disjoint shares into the cache, now each loads the rest
        dist.barrier()
        pairs = {k: pairs[k] if k in pairs else make_pair_device_normals(ctx, k, args.sweeps, args.beams) for k in range(N_SEQUENCE_PAIRS)}
    t_gen = time.perf_counter() - t0
    pairs = [pairs[k] for k in sorted(pairs)]
    if not args.pageable_queue:
        # the scans wait in page-locked memory, as a reader that feeds a GPU would leave them (from pageable arrays every upload is a
        # staged copy on the host thread that drives all three contexts: 283 instead of 291 pairs/s on one GPU)
        pin = lambda a: torch.from_numpy(np.ascontiguousarray(a)).pin_memory().numpy()          # noqa: E731
        pairs = [tuple(synth.Cloud(pin(c.points), pin(c.normals), pin(c.colors)) for c in pr[:2]) + tuple(pr[2:]) for pr in pairs]
    cfg = capi.default_config()
    cfg.metric, cfg.minimizer, cfg.matching, cfg.n_iterations = 1, 0, 0, N_ITER
    cfg.max_distance_sq, cfg.nn_algorithm, cfg.collect_stats = args.max_dist2, 2, 0
    # Three contexts per GPU, each on its own stream: the registrations of different pairs overlap on the device (a single
    # registration is a chain of latency-bound launches that leaves most of the machine idle: 5.0 -> 2.7 ms per pair, measured with
    # profiles/probe_pair_queue.py), and the upload of the next pair overlaps the loops of the others.
    ctxs = [capi.Context(dev.index) for _ in range(3)]
    ms, res, n_mine = None, [], 0
    for rep in range(2):                                   # the first pass warms allocations and graphs
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        # dynamic deal: the ranks draw pair indices from one shared counter (a fresh key per pass), so a rank with cheap pairs takes more
        tickets = parallel.PairTickets(N_SEQUENCE_PAIRS, key=f"icp_bench_pair_queue_pass{rep}") if dynamic else None
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)                                  # the stream is idle: the events bracket the queue, which ends with every
        res = sequence.alignPairs(ctxs, pairs, cfg, tickets=tickets)   # context's stream synchronised (estimate_pose_finish)
        torch.cuda.synchronize()
        e1.record(stream)
        e1.synchronize()
        ms = e0.elapsed_time(e1)
    for c in ctxs:
        c.close()
    done = [r for r in res if r is not None]
    n_mine = len(done)
    print(f"bench: rank {rank}: pair queue: {n_mine} pairs in {ms:.1f} ms ({'dynamic' if dynamic else 'static'} deal)", file=sys.stderr)
    ok = all(r.error is None and r.nIterations == N_ITER for r in done) and (dynamic or n_mine == len(pairs))
    longest = n_mine
    if world > 1:
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
        o = torch.tensor([1 if ok else 0], dtype=torch.int64, device=dev)
        dist.all_reduce(o, op=dist.ReduceOp.MIN)
        ok = bool(o.item())
        c = torch.zeros(world, dtype=torch.int64, device=dev)
        c[rank] = n_mine
        dist.all_reduce(c, op=dist.ReduceOp.SUM)
        counts = [int(x) for x in c.tolist()]
        ok = ok and sum(counts) == N_SEQUENCE_PAIRS           # every pair registered exactly once
        longest = max(counts)
    else:
        counts = [n_mine]
    static_longest = -(-N_SEQUENCE_PAIRS // world)
    return {"pairs": N_SEQUENCE_PAIRS, "n_gpus": world, "pairs_per_s": N_SEQUENCE_PAIRS / (ms * 1e-3), "ms_total": ms,
            "deal": ("dynamic: pair indices drawn from one shared ticket counter (parallel.PairTickets, the process group's store)" if dynamic
                     else "static round-robin (parallel.shard_pairs)"),
            "pairs_per_rank": counts, "pairs_on_the_longest_queue": longest,
            "ideal_speedup_over_one_gpu": N_SEQUENCE_PAIRS / static_longest, "all_pairs_converged_30_iterations": ok,
            "points_per_scan": len(pairs[0][0]) if pairs else None, "scaling": "strong", "collective": "none",
            "path": "sequence.alignPairs: icp_gpu_set_target / set_source (%s host arrays) + icp_gpu_estimate_pose_async / _finish, three contexts (streams) per GPU" % ("pageable" if args.pageable_queue else "page-locked"),
            "input_generation_s_rank0": t_gen}


def sharded_block(torch, dist, capi, ctx, stream, world, rank, dev, args):
    """Config 5b: one 3 M-point pair, the source sharded by points over the ranks (every rank holds the whole target).  Fused: the
    per-iteration all-reduce of the <= 28-double row runs inside reduce_kernel over NVLink peer memory (icp_gpu_peer_*), the loop
    stays one CUDA graph.  Baseline: the same shards with ncclAllReduce on the stream between the two halves of the iteration."""
    from icp_variants_b200 import parallel
    sweeps, beams = args.big_sweeps, args.big_beams
    src, tgt = make_pair_device_normals(ctx, 0, sweeps, beams)
    cfg = capi.default_config()
    cfg.metric, cfg.minimizer, cfg.matching, cfg.n_iterations = 1, 0, 0, N_ITER
    cfg.max_distance_sq, cfg.nn_algorithm, cfg.collect_stats = args.max_dist2, 2, 0
    ctx.set_config(cfg)
    ctx.set_target(tgt.points, tgt.normals, tgt.colors)
    out = {"n_points": int(len(src)), "n_gpus": world, "iterations": N_ITER}

    def timed(fn, reps=3):
        best, res = None, None
        for _ in range(reps):
            torch.cuda.synchronize()
            if world > 1:
                dist.barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            res = fn()
            e1.record(stream)
            e1.synchronize()
            ms = e0.elapsed_time(e1)
            if world > 1:
                t = torch.tensor([ms], dtype=torch.float64, device=dev)
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                ms = float(t.item())
            best = ms if best is None else min(best, ms)
        return best, res

    # one GPU alone (rank 0), whole source: the time the sharded forms are compared with
    pose_single = None
    if rank == 0:
        ctx.set_source(src.points, src.normals, src.colors)
        best = None
        for _ in range(3):
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            pose_single, _, _ = ctx.estimate_pose(want_history=False)
            e1.record(stream); e1.synchronize()
            best = e0.elapsed_time(e1) if best is None else min(best, e0.elapsed_time(e1))
        out["ms_single_gpu"] = best
    if world == 1:
        out["note"] = "N = 1: the unsharded registration (index already built, clouds resident); run with --gpus 2/4/8 for the sharded forms"
        return out
    dist.barrier()
    sl = parallel.shard_points_interleaved(len(src), world, rank)      # uniform subsamples: equal cost per rank and iteration
    ctx.set_source(src.points[sl], src.normals[sl], src.colors[sl])
    # baseline: ncclAllReduce of the row on the stream, no host round trip
    ms_nccl, pose_nccl = timed(lambda: parallel.register_sharded_on_stream(ctx, N_ITER))
    # fused: exchange inside the reduction kernel over peer memory
    parallel.attach_peers(ctx)
    ms_fused, r = timed(lambda: ctx.estimate_pose(want_history=False))
    pose_fused = r[0]
    poses = [None] * world
    dist.all_gather_object(poses, pose_fused.tobytes())
    ctx.peer_detach()
    # what one exchange costs: the same loop on a tiny source (1024 points per rank), attached vs. detached
    tiny = slice(rank * 1024, rank * 1024 + 1024)
    ctx.set_source(src.points[tiny], src.normals[tiny], src.colors[tiny])
    ms_tiny_alone, _ = timed(lambda: ctx.estimate_pose(want_history=False))
    parallel.attach_peers(ctx)
    ms_tiny_fused, _ = timed(lambda: ctx.estimate_pose(want_history=False))
    ctx.peer_detach()
    out.update(ms_fused_peer_memory=ms_fused, ms_nccl_allreduce_on_stream=ms_nccl,
               exchange_bytes_per_iteration_per_peer=27 * 8, exchange_us_per_iteration=(ms_tiny_fused - ms_tiny_alone) * 1e3 / N_ITER,
               pose_identical_on_all_ranks=bool(all(p == poses[0] for p in poses)),
               path="icp_gpu_peer_export / _attach + icp_gpu_estimate_pose (one CUDA graph per rank, exchange inside reduce_kernel)")
    if rank == 0:
        out["speedup_fused_over_single_gpu"] = out["ms_single_gpu"] / ms_fused
        out["speedup_nccl_over_single_gpu"] = out["ms_single_gpu"] / ms_nccl
        out["max_abs_pose_diff_fused_vs_single_gpu"] = float(np.abs(pose_fused - pose_single).max())
        out["max_abs_pose_diff_nccl_vs_single_gpu"] = float(np.abs(pose_nccl - pose_single).max())
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--sweeps", type=int, default=344)
    ap.add_argument("--beams", type=int, default=1077)
    ap.add_argument("--big-sweeps", type=int, default=1720, help="config 5b: sweeps of the point-sharded pair (1720 x 1744 ~ 3 M points)")
    ap.add_argument("--big-beams", type=int, default=1744)
    ap.add_argument("--max-dist2", type=float, default=10.0, help="squared matching distance; alignETH uses 10 (main.cpp:361)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-multi", action="store_true", help="skip the config-5 workloads (pair_queue_44, sharded_3m)")
    ap.add_argument("--static-deal", action="store_true", help="pair_queue_44 with the static round-robin deal at N > 1 (default: shared ticket counter)")
    ap.add_argument("--pageable-queue", action="store_true", help="pair_queue_44 from pageable host arrays (default: page-locked)")
    ap.add_argument("--no-sharded", action="store_true", help="skip sharded_3m only")
    ap.add_argument("--no-flush", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the 4x4 pose each timed arm returned in its last step (rank 0) as DIR/pose.npy "
                         "(device-resident clouds; with --impl reference, the CPU registration) and DIR/pose_e2e.npy (host arrays), float32")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        return run_reference(args)
    args.warmup = max(args.warmup, 3)

    import torch
    import torch.distributed as dist
    from icp_variants_b200 import capi

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (there is no CPU fallback for the icp_gpu_* path)")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)

    src, tgt = make_pair(rank, args.sweeps, args.beams)       # each rank owns its own pair(s): no data-path collective
    ns, nt = len(src), len(tgt)

    ctx = capi.Context(local)
    # One explicit stream for everything: the library's kernels, torch's fills and events, and NCCL's ordering all refer to it
    # (torch's default stream has handle 0, which icp_gpu_set_stream reads as "the context's own stream").
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)
    ctx.set_stream(stream.cuda_stream)                        # torch.cuda.Event only sees torch's current stream
    cfg = capi.default_config()
    cfg.metric, cfg.minimizer, cfg.matching, cfg.n_iterations = 1, 0, 0, N_ITER
    cfg.max_distance_sq = args.max_dist2
    cfg.nn_algorithm = 2
    cfg.collect_stats = 0                                     # work counters cost device atomics: off while timing
    ctx.set_config(cfg)

    # device-resident raw clouds (reference layouts: packed float[3N], uint8[4N])
    d = {k: torch.from_numpy(np.ascontiguousarray(v)).to(dev) for k, v in
         (("sp", src.points), ("sn", src.normals), ("sc", src.colors), ("tp", tgt.points), ("tn", tgt.normals), ("tc", tgt.colors))}
    # pinned host copies for the end-to-end arm
    h = {k: torch.from_numpy(np.ascontiguousarray(v)).pin_memory() for k, v in
         (("sp", src.points), ("sn", src.normals), ("sc", src.colors), ("tp", tgt.points), ("tn", tgt.normals), ("tc", tgt.colors))}
    hn = {k: v.numpy() for k, v in h.items()}
    flush = None if args.no_flush else torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)   # > 126 MB L2

    def step_resident():
        ctx.set_target_dev(d["tp"].data_ptr(), d["tn"].data_ptr(), d["tc"].data_ptr(), nt)
        ctx.set_source_dev(d["sp"].data_ptr(), d["sn"].data_ptr(), d["sc"].data_ptr(), ns)
        return ctx.estimate_pose(want_history=False)

    def step_e2e():
        ctx.set_target(hn["tp"], hn["tn"], hn["tc"])
        ctx.set_source(hn["sp"], hn["sn"], hn["sc"])
        return ctx.estimate_pose(want_history=False)

    def timed(fn, steps, warmup):
        for _ in range(warmup):
            if flush is not None:
                flush.fill_(1)
            fn()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        total_ms, launches, pose = 0.0, 0, None
        for _ in range(steps):
            if flush is not None:
                flush.fill_(1)                                 # L2 flush between timed iterations (outside the events)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            pose, _, n_it = fn()
            e1.record(stream)
            e1.synchronize()
            assert n_it == N_ITER
            total_ms += e0.elapsed_time(e1)
            launches += int(ctx.stats().n_kernel_launches)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            t = torch.tensor([total_ms], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            total_ms = float(t.item())
            l = torch.tensor([launches], dtype=torch.int64, device=dev)
            dist.all_reduce(l, op=dist.ReduceOp.SUM)
            launches = int(l.item())
        return total_ms, launches, pose

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    total_ms, launches, pose = timed(step_resident, args.steps, args.warmup)
    e2e_ms, _, pose_e2e = timed(step_e2e, args.steps, args.warmup)
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"pose": pose, "pose_e2e": pose_e2e})

    # per-kernel timing of the dominant kernel: one extra registration, launch by launch with CUDA events
    ctx.set_target_dev(d["tp"].data_ptr(), d["tn"].data_ptr(), d["tc"].data_ptr(), nt)
    ctx.set_source_dev(d["sp"].data_ptr(), d["sn"].data_ptr(), d["sc"].data_ptr(), ns)
    for _ in range(2):
        _, _, _, tm = ctx.estimate_pose(want_history=False, timings=True)
    # work counters (distance evaluations, staged points, deferred queries): one more, instrumented, registration
    cfg.collect_stats = 1
    ctx.set_config(cfg)
    ctx.set_target_dev(d["tp"].data_ptr(), d["tn"].data_ptr(), d["tc"].data_ptr(), nt)
    ctx.set_source_dev(d["sp"].data_ptr(), d["sn"].data_ptr(), d["sc"].data_ptr(), ns)
    ctx.estimate_pose(want_history=False)
    st = ctx.stats()
    cfg.collect_stats = 0
    ctx.set_config(cfg)
    match_ms = tm.matching_ms / N_ITER
    prep_ms = tm.search_prep_ms / N_ITER
    walk_ms = max(match_ms - prep_ms, 1e-6)          # the search after the fast path: knn_group_kernel + knn_bvh_kernel of one chain (the dominant part)
    solve_ms = tm.solver_ms / N_ITER
    # the FP32 denominators, measured on this device in this run (peak.cu)
    ffma_tflops = ctx.measure_fp32_peak(0)
    nonfma_tflops = ctx.measure_fp32_peak(1)

    line = None
    if rank == 0:
        peak, peak_kind = load_peaks()
        regs = args.steps * world
        value = regs / (total_ms * 1e-3)
        # algorithmic bytes of the fused match kernel per query (SURVEY.md 8d): source point 12 + source normal 12 +
        # matched target point 12 + target normal 12 = 48 B
        alg_bytes = 48.0 * ns
        achieved = alg_bytes / (walk_ms * 1e-3) / 1e9
        evals_per_launch = st.n_distance_evals / N_ITER
        search_tflops = evals_per_launch * 8 / (match_ms * 1e-3) / 1e12
        line = {
            "metric": "icp_registrations_per_s", "value": value, "unit": "reg/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic",
            "config": workload_config(ns, nt, args.max_dist2),
            "ms_per_registration": total_ms / args.steps,
            "mcorr_per_s": (st.n_queries * regs) / (total_ms * 1e-3) / 1e6,
            "e2e": {"value": regs / (e2e_ms * 1e-3), "unit": "reg/s", "ms_per_step": e2e_ms / args.steps,
                    "h2d_bytes_per_step": int((ns + nt) * 28 + 64 + 32 * N_ITER), "d2h_bytes_per_step": int(64 + 16 * 4 * N_ITER + 1024)},
            "gpu_launches": launches,
            "gpu_launches_per_step": launches // max(args.steps * world, 1),
            "roofline": {"kernel": "knn_group_kernel + knn_bvh_kernel<false> (the search after the fast path, timed together: one event pair per iteration)",
                         "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak, "traffic": ncu_traffic("knn_bvh_kernel"), "peak_kind": peak_kind,
                         "algorithmic_bytes_per_launch": alg_bytes, "avg_launch_ms": walk_ms,
                         "note": "issue-bound tree search over L2-resident clouds; see roofline_fp32; traffic = the committed cold-cache capture of knn_bvh_kernel "
                                 "(profiles/r2_ncu_traffic.json, before the group search; with caches as the program leaves them both kernels read < 0.2 MB of DRAM "
                                 "per launch, profiles/r2_ncu_full_search_kernels_group_search.txt)"},
            "roofline_fp32": {"kernels": "knn_prep_kernel (fast path) + knn_group_kernel (runs of deferred neighbours) + knn_bvh_kernel (walk)", "distance_evals_per_launch": evals_per_launch,
                              "gevals_per_s": evals_per_launch / (match_ms * 1e-3) / 1e9, "flop_per_eval": 8, "tflops": search_tflops,
                              "peak_ffma_tflops_measured": ffma_tflops, "peak_fmul_fadd_tflops_measured": nonfma_tflops,
                              "frac_of_measured_non_fma_peak": search_tflops / nonfma_tflops if nonfma_tflops > 0 else None,
                              "frac_of_measured_ffma_peak": search_tflops / ffma_tflops if ffma_tflops > 0 else None,
                              "nodes_per_launch": st.n_nodes_visited / N_ITER, "matched_per_launch": st.n_matched / N_ITER,
                              "note": "contract D1 forbids FMA contraction in the distances: the non-FMA figure is the attainable one"},
            "stage_ms_per_iteration": {"match": match_ms, "match_prep_fast_path": prep_ms, "match_tree_walk": walk_ms, "reduce_solve": solve_ms,
                                       "index_build": tm.index_ms},
            "clocks": clocks,
            "pose_checksum": float(np.abs(pose).sum()),
        }
        if not args.no_cpu_baseline and world == 1:
            line["cpu_baseline"] = cpu_baseline_block(src, tgt, args.max_dist2)
            fl = line["cpu_baseline"].get("flann_like", {})
            if "match_rate_vs_exact" in fl:
                line["flann_match_rate"] = fl["match_rate_vs_exact"][0]
    if not args.no_multi:
        pq = pair_queue_block(torch, dist, capi, ctx, stream, world, rank, dev, args)
        sh = None if args.no_sharded else sharded_block(torch, dist, capi, ctx, stream, world, rank, dev, args)
        if rank == 0:
            line["pair_queue_44"] = pq
            if sh is not None:
                line["sharded_3m"] = sh
    if rank == 0:
        print(json.dumps(line))
    ctx.close()
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
