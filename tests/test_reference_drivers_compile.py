"""Row (b), the drop-in boundary: the reference's OWN drivers -- icp-variants/main.cpp and experiment.cpp, unchanged -- compile as C++14
against include/icp_b200/ (ICPOptimizer.h, NearestNeighbor.h, PointCloud.h, selection.h, weighting.h, constraints.h, ProcrustesAligner.h,
utils.h, ConvergenceMeasure.h, TimeMeasure.h, Eigen.h in place of the reference's headers of the same names).

How: an overlay directory of symbolic links (nothing is copied) -- the drivers and the reference headers the drop-in does not replace
(SimpleMesh.h, the data loaders, VirtualSensor.h ...) next to the drop-in headers -- so that every quoted #include resolves to the
drop-in where one exists.  Third-party headers are the stand-ins of oracle/ref_shim (Eigen, PCL, Ceres) and tests/cpp_shim (FreeImage,
boost::split).  Compile only (-c): the object files would need FreeImage to link and a GPU to run; the running counterpart is
tests/test_cpp_dropin.py (examples/bunny_driver.cpp mirrors main.cpp's bunny path and is compared with the Python binding on the GPU).
CPU only, and only where the reference sources are present (ICP_REFERENCE_ROOT, see oracle/ref.py)."""
import os
import subprocess

import pytest

from oracle import ref as R

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.path.join(R.REFERENCE_ROOT, "icp-variants")
DROPIN = ["ConvergenceMeasure.h", "Eigen.h", "ICPOptimizer.h", "NearestNeighbor.h", "PointCloud.h", "ProcrustesAligner.h", "TimeMeasure.h",
          "constraints.h", "detail.h", "selection.h", "utils.h", "weighting.h"]
KEPT = ["SimpleMesh.h", "BunnyDataLoader.h", "DataLoader.h", "ETHDataLoader.h", "CSVReader.h", "VirtualSensor.h", "FreeImageHelper.h"]

pytestmark = pytest.mark.skipif(not os.path.isdir(REF), reason="the reference sources (ICP_REFERENCE_ROOT/icp-variants) are absent")


@pytest.fixture(scope="module")
def overlay(tmp_path_factory):
    top = tmp_path_factory.mktemp("dropin_overlay")
    inc = top / "icp_b200"
    inc.mkdir()
    os.symlink(os.path.join(ROOT, "include", "icp_gpu.h"), top / "icp_gpu.h")
    for h in DROPIN:
        os.symlink(os.path.join(ROOT, "include", "icp_b200", h), inc / h)
    for h in KEPT + ["main.cpp", "experiment.cpp"]:
        os.symlink(os.path.join(REF, h), inc / h)
    return inc


def test_the_dropin_replaces_every_header_of_the_path():
    # every header of the reference that is on the registration path has a drop-in of the same name
    for h in ("ICPOptimizer.h", "NearestNeighbor.h", "selection.h", "weighting.h", "constraints.h", "ProcrustesAligner.h", "utils.h", "PointCloud.h",
              "ConvergenceMeasure.h", "TimeMeasure.h", "Eigen.h"):
        assert os.path.exists(os.path.join(REF, h)) and os.path.exists(os.path.join(ROOT, "include", "icp_b200", h)), h


@pytest.mark.parametrize("driver", ["main.cpp", "experiment.cpp"])
def test_reference_driver_compiles_unchanged_against_the_dropin_headers(overlay, driver):
    obj = overlay / (driver + ".o")
    cmd = ["g++", "-std=c++14", "-c", "-w", "-DICP_B200_USE_EIGEN", "-I", str(overlay), "-I", os.path.join(ROOT, "oracle", "ref_shim"),
           "-I", os.path.join(ROOT, "tests", "cpp_shim"), str(overlay / driver), "-o", str(obj)]
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    assert r.returncode == 0, r.stdout[-6000:]
    # the object file references the drop-in's C ABI, i.e. the drop-in classes were the ones compiled
    syms = subprocess.run(["nm", "-C", "--undefined-only", str(obj)], stdout=subprocess.PIPE, text=True).stdout
    assert "icp_gpu_estimate_pose" in syms and "icp_gpu_set_target" in syms
    assert "flann" not in syms.lower() and "ceres::Solve" not in syms
