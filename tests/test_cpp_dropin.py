"""The C++14 drop-in headers (include/icp_b200/*.h: the reference's ICPOptimizer / NearestNeighborSearch
class names and signatures over the icp_gpu_* C ABI): they compile as C++14 and link against the library
(CPU), and a reference-style driver gives the same pose as the Python binding (GPU)."""
import os
import subprocess

import numpy as np
import pytest

from icp_variants_b200 import capi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def build_driver(out_dir):
    capi.build()
    libdir = os.path.dirname(capi.LIB_PATH)
    exe = str(out_dir / "icp_b200_bunny_driver")
    cmd = ["g++", "-std=c++14", "-Wall", "-Wextra", "-Werror", "-I", os.path.join(ROOT, "include"),
           os.path.join(ROOT, "examples", "bunny_driver.cpp"), "-o", exe, "-L", libdir, "-licp_gpu", f"-Wl,-rpath,{libdir}"]
    subprocess.run(cmd, check=True)
    return exe


def build_nn_check(out_dir):
    """The matcher classes alone, as a reference user would instantiate them."""
    src = '#include "icp_b200/NearestNeighbor.h"\nint main(){ NearestNeighborSearchFlann f; NearestNeighborSearchProjective p; NearestNeighborSearchBruteForce b; f.setMatchingMaxDistance(0.1f); return (int)f.queryMatches({}).size(); }\n'
    libdir = os.path.dirname(capi.LIB_PATH)
    exe = str(out_dir / "icp_b200_nn_check")
    subprocess.run(["g++", "-std=c++14", "-x", "c++", "-", "-I", os.path.join(ROOT, "include"), "-o", exe,
                    "-L", libdir, "-licp_gpu", f"-Wl,-rpath,{libdir}"], input=src, text=True, check=True)
    return exe


def test_dropin_headers_compile_as_cpp14(tmp_path):
    build_driver(tmp_path)
    build_nn_check(tmp_path)


def test_driver_without_gpu_reports_and_does_not_hang(tmp_path):
    if capi.lib().icp_gpu_device_count() > 0:
        pytest.skip("a GPU is present")
    exe = build_driver(tmp_path)
    r = subprocess.run([build_nn_check(tmp_path)], stdout=subprocess.PIPE, text=True, timeout=60)
    assert "no usable CUDA device" in r.stdout and r.returncode == 0
    assert os.path.exists(exe)


def _dump(path, cloud):
    with open(path, "wb") as f:
        f.write(np.int32(len(cloud.points)).tobytes())
        f.write(np.ascontiguousarray(cloud.points, np.float32).tobytes())
        f.write(np.ascontiguousarray(cloud.normals, np.float32).tobytes())


@pytest.mark.gpu
@pytest.mark.parametrize("linear,metric", [(1, 0), (1, 1), (1, 2), (0, 1)])
def test_cpp_driver_matches_python_binding(bunny, linear, metric, tmp_path):
    src, tgt, _, _ = bunny
    exe = build_driver(tmp_path)
    src_bin, tgt_bin = str(tmp_path / "src.bin"), str(tmp_path / "tgt.bin")
    _dump(src_bin, src)
    _dump(tgt_bin, tgt)
    r = subprocess.run([exe, src_bin, tgt_bin, str(linear), str(metric), "20"],
                       stdout=subprocess.PIPE, text=True, check=True, timeout=120)
    line = [l for l in r.stdout.splitlines() if l.startswith("POSE")][0]
    pose_cpp = capi.pose_from_c(np.array(line.split()[1:], np.float32))
    with capi.Context(0) as c:
        cfg = capi.default_config()
        cfg.metric, cfg.minimizer, cfg.n_iterations, cfg.max_distance_sq = metric, 0 if linear else 1, 20, 0.0003
        c.set_config(cfg)
        c.set_target(tgt.points, tgt.normals, tgt.colors)
        c.set_source(src.points, src.normals, src.colors)
        pose_py, _, _ = c.estimate_pose()
    assert np.allclose(pose_cpp, pose_py, rtol=0, atol=1e-7)
    # ConvergenceMeasure filled from the device (icp_gpu_convergence_errors): main.cpp:105-120's 4 correspondences
    from oracle import oracle as orc
    _, _, gs, gt = bunny
    f = [l for l in r.stdout.splitlines() if l.startswith("RMSE")][0].split()
    assert int(f[5]) == 20
    assert float(f[1]) == pytest.approx(orc.rmse(pose_py, src.points[gs], tgt.points[gt]), rel=1e-6)
    assert float(f[3]) == pytest.approx(orc.benchmark_error(pose_py, src.points[gs], tgt.points[gt]), rel=1e-6)


def build_value_driver(out_dir):
    capi.build()
    libdir = os.path.dirname(capi.LIB_PATH)
    exe = str(out_dir / "icp_b200_value_driver")
    cmd = ["g++", "-std=c++14", "-Wall", "-Wextra", "-Werror", "-I", os.path.join(ROOT, "include"),
           os.path.join(ROOT, "examples", "value_classes_driver.cpp"), "-o", exe, "-L", libdir, "-licp_gpu", f"-Wl,-rpath,{libdir}"]
    subprocess.run(cmd, check=True)
    return exe


def test_value_classes_compile_as_cpp14(tmp_path):
    build_value_driver(tmp_path)


def _fingerprint(a):
    u = np.ascontiguousarray(a, np.float32).view(np.uint32).reshape(-1).astype(np.uint64)
    k = (2 * np.arange(len(u), dtype=np.uint64) + 1)
    return int((u * k).sum(dtype=np.uint64))


@pytest.mark.gpu
def test_value_classes_driver_equals_oracle(bunny, tmp_path):
    """PointSelection, WeightingMethod, the three functors, ProcrustesAligner, PoseIncrement, transformPoints / transformNormals,
    PointCloud::change_pose and ConvergenceMeasure as a C++ user of the reference holds them -- each a thin class over an icp_gpu_* call
    (include/icp_b200/) -- against the oracle: bit-exact transforms / matches / weights, 1e-5 poses, the functor values to 1e-12."""
    from oracle import oracle as orc
    src, tgt, _, _ = bunny
    exe = build_value_driver(tmp_path)
    src_bin, tgt_bin = str(tmp_path / "src.bin"), str(tmp_path / "tgt.bin")
    _dump(src_bin, src)
    _dump(tgt_bin, tgt)
    r = subprocess.run([exe, src_bin, tgt_bin], stdout=subprocess.PIPE, text=True, check=True, timeout=120)
    out = {l.split()[0]: l.split()[1:] for l in r.stdout.splitlines() if l and l.split()[0].isupper()}
    pose = capi.pose_from_c(np.array(out["POSE"], np.float32))
    x = np.array([0.01, -0.02, 0.03, 0.001, 0.002, -0.001])
    th = np.linalg.norm(x[:3]); K = np.array([[0, -x[2], x[1]], [x[2], 0, -x[0]], [-x[1], x[0], 0]])
    Rm = np.eye(3) + np.sin(th) / th * K + (1 - np.cos(th)) / th ** 2 * K @ K
    assert np.allclose(pose[:3, :3], Rm, atol=1e-7) and np.allclose(pose[:3, 3], x[3:], atol=1e-9)
    q, qn = orc.transform_points(pose, src.points), orc.transform_normals(pose, src.normals)
    assert [int(v) for v in out["TRANSFORM"]] == [_fingerprint(q), _fingerprint(qn)]
    assert int(out["CHANGEPOSE"][0]) == _fingerprint(q)
    m = orc.KdTree(tgt.points).query(q, 0.0003)
    m = orc.apply_weights(1, 0.0003, q, qn, src.colors, tgt.points, tgt.normals, tgt.colors, m)
    keep = m["idx"] >= 0
    assert int(out["MATCH"][0]) == int(keep.sum()) and int(out["MATCH"][1]) == int(m["idx"][keep].sum())
    assert float(out["MATCH"][2]) == pytest.approx(float(m["weight"][keep].astype(np.float64).sum()), rel=1e-7)
    rc, p2p = orc.solve_p2p(q[keep], tgt.points[m["idx"][keep]], m["weight"][keep])
    got = capi.pose_from_c(np.array(out["PROCRUSTES"], np.float32))
    assert rc == 0 and np.abs(got - p2p).max() < 1e-5
    rng = orc.MT19937(); rng.seed(42)
    sel = [i for i in range(len(src.points)) if rng.canonical() < np.float32(0.25)]
    assert int(out["SELECTION"][0]) == len(sel) and int(out["SELECTION"][1]) == sum(sel)
    # the functors: closed forms of constraints.h
    s0, d0, ns0, nt0 = (a.astype(np.float64) for a in (src.points[0], tgt.points[0], src.normals[0], tgt.normals[0]))
    w = np.float64(np.float32(0.7)); y = Rm @ s0 + x[3:]
    exp = list(np.float64(np.float32(0.1)) * w * (y - d0)) + [w * (nt0 @ (y - d0)), w * ((nt0 + ns0) @ (y - Rm.T @ d0))]
    assert np.allclose([float(v) for v in out["FUNCTORS"]], exp, rtol=0, atol=1e-12)
    assert float(out["ERRORS"][0]) == pytest.approx(orc.rmse(pose, src.points[:64], tgt.points[:64]), rel=2e-6)
    assert float(out["ERRORS"][1]) == pytest.approx(orc.benchmark_error(pose, src.points[:64], tgt.points[:64]), rel=1e-9)
