"""ctypes front-end of tests/voxel_reference.c, the CPU restatement of the device's voxel-grid downsampling (DESIGN.md section 4, V1-V5).

TEST INFRASTRUCTURE ONLY -- imported by tests/test_gpu_voxel.py, tests/test_voxel_reference.py and profiles/measure_voxel.py.  The
library is compiled on first use into the system's temporary directory (keyed by the source's hash), never into the repository."""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

_SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "voxel_reference.c")
_lib = None


def lib():
    global _lib
    if _lib is None:
        with open(_SRC, "rb") as f:
            digest = hashlib.sha1(f.read()).hexdigest()[:16]
        so = os.path.join(tempfile.gettempdir(), f"icp_voxel_reference_{os.getuid()}_{digest}.so")
        if not os.path.exists(so):
            cc = os.environ.get("CC", "cc")
            tmp = f"{so}.{os.getpid()}.tmp"
            subprocess.run([cc, "-std=c11", "-O2", "-ffp-contract=off", "-fno-fast-math", "-fPIC", "-shared", "-o", tmp, _SRC, "-lm"], check=True)
            os.replace(tmp, so)
        _lib = C.CDLL(so)
    return _lib


def _f32(a):
    return None if a is None else np.ascontiguousarray(a, np.float32).reshape(-1, 3)


def _u8(a):
    return None if a is None else np.ascontiguousarray(a, np.uint8).reshape(-1, 4)


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def voxel_downsample(pts, voxel_size, nrm=None, rgba=None, off=None):
    """(points, normals or None, colours or None, offsets [B+1]) of the concatenated clouds pts (off None: one cloud), cloud b's voxels
    at [off_out[b], off_out[b+1])."""
    pts, nrm, rgba = _f32(pts), _f32(nrm), _u8(rgba)
    off = np.array([0, len(pts)], np.int64) if off is None else np.ascontiguousarray(off, np.int64)
    B = len(off) - 1
    po = np.empty((max(len(pts), 1), 3), np.float32)
    no = np.empty((max(len(pts), 1), 3), np.float32) if nrm is not None else None
    co = np.empty((max(len(pts), 1), 4), np.uint8) if rgba is not None else None
    oo = np.zeros(B + 1, np.int64)
    rc = lib().vref_voxel_downsample(C.c_int32(B), _p(pts), _p(nrm), _p(rgba), _p(off), C.c_float(voxel_size), _p(po), _p(no), _p(co), _p(oo))
    if rc != 0:
        raise ValueError(f"voxel_downsample: cloud {-rc - 1} has a voxel index outside int32")
    m = int(oo[-1])
    return po[:m].copy(), None if no is None else no[:m].copy(), None if co is None else co[:m].copy(), oo
