"""CPU-side checks of the drop-in boundary: the C-ABI library builds, loads, exports every symbol
include/icp_gpu.h declares, and refuses to run without a GPU (no CPU fallback)."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from icp_variants_b200 import capi


@pytest.fixture(scope="module")
def lib():
    capi.build()
    return capi.lib()


def test_library_exports_every_declared_symbol(lib):
    names = capi.declared_symbols()
    assert len(names) >= 28
    for n in names:
        assert hasattr(lib, n), f"{n} declared in include/icp_gpu.h but not exported"
    out = subprocess.run(["nm", "-D", "--defined-only", capi.LIB_PATH], stdout=subprocess.PIPE, text=True, check=True).stdout
    exported = sorted(l.split()[-1] for l in out.splitlines() if " T " in l)
    assert exported == names, "the library must export exactly the C ABI"


def test_abi_version_and_default_config(lib):
    assert lib.icp_gpu_abi_version() == 4
    c = capi.default_config()
    # ICPOptimizer constructor defaults, ICPOptimizer.h:29-31
    assert (c.metric, c.selection, c.rejection, c.weighting, c.n_iterations, c.matching) == (0, 0, 1, 0, 20, 0)
    assert abs(c.max_distance_sq - 0.0003) < 1e-9 and c.color_icp == 0 and c.multires == 0 and c.lm_max_iterations == 10


def test_config_struct_layout_matches_header(tmp_path):
    """sizeof(icp_gpu_config) as the C compiler sees it == the ctypes mirror."""
    src = '#include "icp_gpu.h"\n#include <stdio.h>\nint main(){printf("%zu %zu %zu", sizeof(icp_gpu_config), sizeof(icp_gpu_timings), sizeof(icp_gpu_stats));return 0;}'
    exe = str(tmp_path / "icp_gpu_sizeof")
    subprocess.run(["gcc", "-x", "c", "-", "-I", os.path.dirname(capi.HEADER_PATH), "-o", exe], input=src, text=True, check=True)
    sizes = [int(x) for x in subprocess.run([exe], stdout=subprocess.PIPE, text=True, check=True).stdout.split()]
    assert sizes == [C.sizeof(capi.Config), C.sizeof(capi.Timings), C.sizeof(capi.Stats)]


def test_no_cpu_fallback(lib):
    if lib.icp_gpu_device_count() > 0:
        pytest.skip("a GPU is present")
    with pytest.raises(capi.IcpGpuError) as e:
        capi.Context(0)
    assert e.value.code == capi.E_CUDA


def test_pose_layout_roundtrip():
    p = np.arange(16, dtype=np.float32).reshape(4, 4)
    v = capi.pose_to_c(p)
    assert v[12] == p[0, 3] and v[1] == p[1, 0]       # column-major like Eigen::Matrix4f::data()
    assert np.array_equal(capi.pose_from_c(v), p)


def test_header_constants_match_the_python_mirror(tmp_path):
    """Error codes and the peer-exchange constants as the C compiler sees them == capi.py."""
    src = ('#include "icp_gpu.h"\n#include <stdio.h>\nint main(){printf("%d %d %d %d %d %d %d %d %d", ICP_GPU_E_CUDA, ICP_GPU_E_ARG, ICP_GPU_E_STATE, '
           'ICP_GPU_E_NO_MATCHES, ICP_GPU_E_NUMERIC, ICP_GPU_E_PEER, ICP_GPU_MAX_PEERS, ICP_GPU_PEER_HANDLE_BYTES, ICP_GPU_MAX_PARTIALS);return 0;}')
    exe = str(tmp_path / "icp_gpu_consts")
    subprocess.run(["gcc", "-x", "c", "-", "-I", os.path.dirname(capi.HEADER_PATH), "-o", exe], input=src, text=True, check=True)
    vals = [int(x) for x in subprocess.run([exe], stdout=subprocess.PIPE, text=True, check=True).stdout.split()]
    assert vals == [capi.E_CUDA, capi.E_ARG, capi.E_STATE, capi.E_NO_MATCHES, capi.E_NUMERIC, capi.E_PEER, capi.MAX_PEERS,
                    capi.PEER_HANDLE_BYTES, capi.MAX_PARTIALS]
