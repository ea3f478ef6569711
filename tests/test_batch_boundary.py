"""CPU-side checks of the batched-registration boundary: the header's target cap equals the Python mirror, and the host
helpers lay B clouds out as the C ABI reads them (concatenated points, B+1 offsets, column-major poses)."""
import os
import subprocess

import numpy as np
import pytest

from icp_variants_b200 import capi, synth


def test_batch_cap_matches_the_header(tmp_path):
    src = '#include "icp_gpu.h"\n#include <stdio.h>\nint main(){printf("%d", ICP_GPU_BATCH_MAX_TARGET);return 0;}'
    exe = str(tmp_path / "icp_gpu_batch_cap")
    subprocess.run(["gcc", "-x", "c", "-", "-I", os.path.dirname(capi.HEADER_PATH), "-o", exe], input=src, text=True, check=True)
    assert int(subprocess.run([exe], stdout=subprocess.PIPE, text=True, check=True).stdout) == capi.BATCH_MAX_TARGET
    assert {"icp_gpu_estimate_pose_batch", "icp_gpu_estimate_pose_batch_dev"} <= set(capi.declared_symbols())


def test_concatenated_clouds_and_offsets():
    a = synth.Cloud(np.arange(6, dtype=np.float32).reshape(2, 3), np.ones((2, 3), np.float32), None)
    b = np.full((3, 3), 7.0, np.float32)                       # a bare point array: zero normals
    e = np.zeros((0, 3), np.float32)
    xyz, nrm, off = capi._concat_clouds([a, e, b])
    assert off.dtype == np.int64 and off.tolist() == [0, 2, 2, 5]
    assert np.array_equal(xyz[:2], a.points) and np.array_equal(xyz[2:], b)
    assert np.array_equal(nrm[:2], a.normals) and not nrm[2:].any()
    assert capi._concat_clouds([b, e])[1] is None                # no cloud has normals: none are passed
    with pytest.raises(ValueError):
        capi._concat_clouds([synth.Cloud(np.zeros((2, 3), np.float32), np.zeros((1, 3), np.float32), None)])


def test_batch_poses_are_column_major():
    p = np.arange(32, dtype=np.float32).reshape(2, 4, 4)
    c = capi._batch_poses(p, 2)
    assert c.shape == (2, 16) and np.array_equal(c[1], capi.pose_to_c(p[1]))
    assert np.array_equal(capi._batch_poses(None, 3), np.tile(capi.pose_to_c(np.eye(4)), (3, 1)))
    with pytest.raises(ValueError):
        capi._batch_poses(p, 3)
